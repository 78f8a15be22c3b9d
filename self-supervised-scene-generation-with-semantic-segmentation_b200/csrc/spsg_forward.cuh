// spsg_forward.cuh -- the persistent forward kernel (march, refinement, write-out, fused 2D losses) and the loss finalisation.
// Fragment of libspsg_raycast.so: included by spsg_raycast.cu INSIDE its anonymous namespace, in the order listed there
// (one translation unit; every device function is inlined into the kernels that use it).
#pragma once

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------

#ifdef SPSG_STATS
// development build only (-DSPSG_STATS): event counters of the march, read back with spsg_debug_stats()
__device__ unsigned long long g_stats[48];
__device__ int g_tile_stats[131072][8];  // per tile: total, setup, march, refine, epilogue cycles, iterations, smid, start
#define STAT_MAX(k, v) atomicMax(&g_stats[k], (unsigned long long)(v))
#define STAT_ADD(k, v) atomicAdd(&g_stats[k], (unsigned long long)(v))
#if SPSG_STATS == 1
#define EVT_ADD(k, v) STAT_ADD(k, v)  // per-event counters (slow: perturbs timing)
#else
#define EVT_ADD(k, v)
#endif
#else
#define STAT_ADD(k, v)
#define STAT_MAX(k, v)
#define EVT_ADD(k, v)
#endif

struct LossArgs {
    const float *target_depth, *target_color, *weight_color;
    const uint8_t *target_label;
    const float *class_weight;
    float voxelsize;
    double *accum;  // [0]=sum|d-t| [1]=#depth [2]=sum|c-t| [3]=#colour elems [4]=sum w*nll [5]=sum w
    // forward only: the CTA that finishes last reduces the accumulators into loss_out (no finalize launch)
    float *loss_out;
    int32_t *done;  // CTAs finished (zeroed per call)
    float w_depth, w_color, w_sem;
    int sem_channels;  // C of the kGenericSem kernels (in the struct's tail padding: no kernel parameter offset moves)
};

__device__ __forceinline__ void finalize_loss_warp(const double *acc, float *__restrict__ out, float w_depth, float w_color,
                                                   float w_sem, bool has_depth, bool has_color, bool has_sem, int lane);

struct ForwardArgs {
    const int32_t *sparse_mapping;
    const float *vals_sdf, *vals_color, *vals_normal, *vals_semantic;
    const float *view_matrix, *intrinsics;
    float *image_color, *image_depth, *image_normal, *image_semantic;
    int32_t *mapping3dto2d, *mapping3dto2d_num;
    const float *dense;
    const uint2 *vbits;   // [B][vpc]
    const uint8_t *bmap;  // [B][bpc]
    size_t vpc, bpc;
    int wpr;
    int maps_in_smem;
    int32_t *tile_counter;  // [B], zeroed per call
    int32_t *list_count;
    int2 *list;
    int32_t *hits;
    int width, height;
    float depth_min, depth_max, thresh, inc;
    int dimx, dimy, dimz;
    int vx, vy, vz;  // samples with floor(p) in [0, v) per axis can be valid: dim - 1, or 0 when the maps are not in use
    int nbx, nby, nbz;
    int num_chunks, views, max_pixels;
    long long num_locs;
    unsigned flags;
    int vec_ok;  // image rows 16-byte aligned: float4 write-out allowed
    float guard; // see frac_guard
    LossArgs loss;
    spsg_grad_buffers clear;  // gradient rows [0, clear_rows) to zero for the backward that follows (or clear_rows = 0)
    long long clear_rows;
    // kLabels (spsg_raycast_labels), after every other field so that no kernel parameter offset moves: uint8 label per
    // voxel in, uint8 label per pixel out, optional C + 1 counters (C = loss.sem_channels)
    const uint8_t *voxel_labels;
    uint8_t *image_label;
    unsigned long long *hist;
    // kEval (spsg_raycast_eval), after the kLabels fields (voxel_labels = predicted label per voxel, image_label = optional
    // per-pixel output): optional (C + 1)^2 confusion counters, and 8 floats per (image, tile) for the six loss partials
    unsigned long long *confusion;
    float *eval_tiles;
};

constexpr int kTileW = 16, kTileH = 8;  // pixels per CTA of the occupancy kernel: 4 warps of 8x4 pixels
constexpr int kTilePix = kTileW * kTileH;

constexpr int kWarpW = 8, kWarpH = 4;                   // pixels per warp tile
constexpr int kFwdWarps = 24;                           // warps of the persistent forward CTA (one CTA per SM)
#ifndef SPSG_FWD_WARPS_LARGE
#define SPSG_FWD_WARPS_LARGE 28
#endif
constexpr int kFwdWarpsLarge = SPSG_FWD_WARPS_LARGE;                      // ... for launches with many tiles per SM (more latency hiding, a few spills)
constexpr int kFwdThreads = kFwdWarps * 32;
constexpr int kStageFloats = 14 * 32;                   // per-warp write-out staging: the widest channel group
__host__ __device__ constexpr size_t fwd_smem_fixed(int warps) { return 128 + (size_t)warps * kStageFloats * sizeof(float); }
constexpr size_t kFwdSmemFixed = fwd_smem_fixed(kFwdWarpsLarge);  // residency test uses the larger CTA
constexpr size_t kFwdSmemMax = 232448 - 1024;           // 227 KB opt-in limit per CTA, minus the static shared memory

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- TMA bulk copy global -> shared, completion on an mbarrier (sm_90+ PTX)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned phase) {
    unsigned done;
    do {
        asm volatile(
            "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
    } while (!done);
}

// Write-out of one channel group of a warp's 8x4 pixel tile: smem [kWarpH][kWarpW*C] -> global rows, by the warp.
// `pix0` = global pixel index of the tile's first pixel (image * H * W + y0 * W + x0).
template <int C>
__device__ __forceinline__ void store_warp_tile(const float *__restrict__ s, float *__restrict__ g, size_t pix0, int x0,
                                                int y0, int width, int height, bool vec, int lane) {
    const int rows = min(kWarpH, height - y0), cols = min(kWarpW, width - x0);
    constexpr int kRow = kWarpW * C;
    if (rows <= 0 || cols <= 0) return;
    float *__restrict__ base = g + pix0 * C;
    const int stride = width * C;  // floats between image rows (< 2^31: checked on the host)
    if (vec && cols == kWarpW) {
        constexpr int kVecRow = kRow / 4;
        // the staged rows are contiguous: element e of the tile is float4 e of the staging buffer
#pragma unroll 1
        for (int e = lane; e < rows * kVecRow; e += 32) {
            const int r = e / kVecRow, k = e - r * kVecRow;
            __stcs(reinterpret_cast<float4 *>(base + r * stride) + k, reinterpret_cast<const float4 *>(s)[e]);
        }
    } else {
        const int n = cols * C;
#pragma unroll 1
        for (int e = lane; e < rows * kRow; e += 32) {
            const int r = e / kRow, k = e - r * kRow;
            if (k < n) __stcs(base + r * stride + k, s[e]);
        }
    }
}

// Write-out of the C-channel semantic rows of a warp's 8x4 pixel tile (kGenericSem).  Each tile row is 8*C contiguous
// floats of the image; lane l writes floats l, l + 32, ... of it, taking the pixel's hit voxel from its lane by shuffle and
// the value from that voxel's payload row.  Every store instruction covers 128 contiguous bytes, so unlike the 14-channel
// path no staging is needed, and no payload is held in registers.  Loop bounds are uniform over the warp (the shuffles).
__device__ __forceinline__ void store_semantic_rows(const float *__restrict__ vals, int C, int hit, float *__restrict__ g,
                                                    size_t pix0, int x0, int y0, int width, int height, int lane) {
    const int rows = min(kWarpH, height - y0), cols = min(kWarpW, width - x0);
    if (rows <= 0 || cols <= 0) return;
    const int n = cols * C;
    float *__restrict__ base = g + pix0 * C;
    const size_t stride = (size_t)width * C;
#pragma unroll 1
    for (int r = 0; r < rows; r++) {
#pragma unroll 1
        for (int k0 = 0; k0 < n; k0 += 32) {
            const int k = k0 + lane, px = min(k / C, kWarpW - 1);
            const int h = __shfl_sync(0xffffffffu, hit, r * kWarpW + px);
            if (k < n) __stcs(base + r * stride + k, h >= 0 ? __ldg(vals + (size_t)h * C + (k - px * C)) : -CUDART_INF_F);
        }
    }
}

// Cross-entropy of one pixel over the C logits of row l (kGenericSem): max, sum of exp(l_k - max) in k order, log, in the
// order of the 14-channel code it stands beside (kFast: __expf / __logf as the fused forward, else expf / logf as the
// stand-alone losses).
template <bool kFast>
__device__ __forceinline__ float ce_nll(const float *__restrict__ l, int C, int y) {
    float m = __ldg(l);
#pragma unroll 1
    for (int k = 1; k < C; k++) m = fmaxf(m, __ldg(l + k));
    float s = 0.0f;
#pragma unroll 1
    for (int k = 0; k < C; k++) s += kFast ? __expf(__ldg(l + k) - m) : expf(__ldg(l + k) - m);
    return (kFast ? __logf(s) : logf(s)) + m - __ldg(l + y);
}

// words [0, n) of p := 0, this warp's share of a launch-wide sweep: 16-byte stores where p is aligned
__device__ __forceinline__ void clear_span(float *__restrict__ p, size_t n, size_t warp_id, size_t num_warps, int lane) {
    if ((reinterpret_cast<uintptr_t>(p) & 15u) == 0) {
        const size_t n4 = n >> 2;
        float4 *p4 = reinterpret_cast<float4 *>(p);
        for (size_t i = warp_id * 32 + lane; i < n4; i += num_warps * 32) p4[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (warp_id == 0 && lane < (int)(n & 3)) p[(n4 << 2) + lane] = 0.0f;
    } else {
        for (size_t i = warp_id * 32 + lane; i < n; i += num_warps * 32) p[i] = 0.0f;
    }
}

// Persistent forward: one CTA per SM, one thread per ray, one 8x4-pixel tile per warp at a time.
// kernel.cu:265-297 (init + ray), :190-263 (march), :166-187 (regula falsi), :215-249 (hit write-out + voxel->pixel
// registration); kLoss adds the 2D losses (train.py:635-638, loss.py:246-257, train.py:744-746) to the epilogue.
// CTA i works on chunk i % B (then i % B + gridDim, ...): the chunk's cell-class bit planes and block map are pulled
// into shared memory once by TMA bulk copies, so the march's "does this sample need arithmetic" lookups never leave
// the SM; tiles of the chunk's images are dealt to warps first statically, then from a global counter.
// kViewNormals (SPSG_FLAG_VIEW_NORMALS, several views): vals_normal is (N,F,3) and image chunk*F + f reads row (hit, f); the
// backward's normal rows to clear are N*F.
// kGenericSem (C != 14, or SPSG_FLAG_GENERIC_SEMANTIC): vals_semantic / image_semantic hold a.loss.sem_channels channels; the
// semantic rows are written by store_semantic_rows and the fused cross-entropy reads the hit voxel's payload row.  The
// march, the registration and every other rendering are the same code.
// kLabels (spsg_raycast_labels): the same march, then an epilogue that writes one byte per pixel -- the hit voxel's
// label, min(voxel_labels[hit], C), or C on a miss -- and, with a.hist, counts pixels per label in a shared-memory
// histogram (the staging area, which this epilogue does not use) flushed once per CTA with integer atomics.  No payload
// loads, no float image, no registration, no work list, no hit records, no gradient rows.
// kEval (spsg_raycast_eval): the same march, then an epilogue for evaluation without a backward: the predicted label of
// the pixel (as kLabels, from voxel_labels), optionally stored; the (C + 1)^2 confusion of min(target label, C) against it,
// counted in shared memory (the staging area) and flushed once per CTA with integer atomics; and the three 2D loss terms
// with kLoss's per-pixel arithmetic (the C-generic cross-entropy at every C), whose six per-warp partials go to the tile's
// own slot of a.eval_tiles for eval_loss_sum_kernel to add in a fixed order.  Reads the hit voxel's colour and logits, no
// normals; no float atomics, no image, registration, work list or hit records.
template <bool kLoss, bool kSmemMaps, int kWarps, bool kViewNormals, bool kGenericSem = false, bool kLabels = false,
          bool kEval = false>
__global__ void __launch_bounds__(kWarps * 32, 1) raycast_forward_kernel(const ForwardArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ float4 s_steps[kStepEntries];
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *stage = reinterpret_cast<float *>(smem + 128) + warp * kStageFloats;
    uint2 *s_vbits = reinterpret_cast<uint2 *>(smem + fwd_smem_fixed(kWarps));
    uint8_t *s_bmap = reinterpret_cast<uint8_t *>(s_vbits + a.vpc);
    const unsigned kFull = 0xffffffffu;
    const float kInf = CUDART_INF_F;

    if (!kLabels && !kEval && a.clear_rows > 0) {
        // The backward's output rows are zeroed here (the reference memsets its whole d_* buffers, kernel.cu:557-560): a few
        // fire-and-forget stores per warp that overlap the march, instead of a longer fill pass in front of the index build.
        const size_t wid = (size_t)blockIdx.x * kWarps + warp, nw = (size_t)gridDim.x * kWarps, n = (size_t)a.clear_rows;
        clear_span(a.clear.d_semantic, n * (kGenericSem ? (size_t)a.loss.sem_channels : 14), wid, nw, lane);
        clear_span(a.clear.d_color, n * 3, wid, nw, lane);
        clear_span(a.clear.d_normal, n * 3 * (kViewNormals ? (size_t)a.views : 1), wid, nw, lane);
        clear_span(a.clear.d_depth, n, wid, nw, lane);
    }
    if (threadIdx.x < kStepEntries) step_table_fill(s_steps, threadIdx.x, a.inc);
    if (kSmemMaps && threadIdx.x == 0) mbar_init(mbar, 1);
    if (kLabels && a.hist && threadIdx.x <= a.loss.sem_channels) reinterpret_cast<unsigned *>(smem + 128)[threadIdx.x] = 0u;
    const int conf_cells = (a.loss.sem_channels + 1) * (a.loss.sem_channels + 1);  // (kEval)
    if (kEval && a.confusion)
        for (int i = threadIdx.x; i < conf_cells; i += kWarps * 32) reinterpret_cast<unsigned *>(smem + 128)[i] = 0u;
    __syncthreads();
    unsigned phase = 0;
    const float inv_inc = rcp_approx(a.inc);

    const size_t cells = (size_t)a.dimz * a.dimy * a.dimx;
    const bool clip = !(a.flags & SPSG_FLAG_NO_CLIP);
    const bool skip = !(a.flags & SPSG_FLAG_NO_BRICK_SKIP);
    const bool fast_ok = max(a.dimx, max(a.dimy, a.dimz)) <= kMaxFastDim;
    const bool skip_ok = skip && fast_ok;
    // warp tiles are numbered so that the four tiles of a 16x8 pixel block are consecutive
    const int tiles_x = (a.width + kWarpW - 1) / kWarpW, tiles_y = (a.height + kWarpH - 1) / kWarpH;
    const int blocks_x = (tiles_x + 1) >> 1, blocks_y = (tiles_y + 1) >> 1;
    const int tiles_per_image = blocks_x * blocks_y * 4;
    const int total_tiles = tiles_per_image * a.views;

    // Chunks of this CTA: its own first (chunk i % B, then + gridDim, ...), then -- work stealing for ragged batches --
    // any other chunk that still has unclaimed tiles in its dynamic counter.  Warp 0 picks, the CTA follows.
    __shared__ int s_next_chunk;
    int own_next = blockIdx.x % a.num_chunks, steal_k = 0;
    for (bool first_chunk = true;; first_chunk = false) {
        // Maps read through L1 (!kSmemMaps): nothing ties a CTA to a chunk, so there is one pass in which every warp takes
        // tiles of ALL chunks from one global counter (chunk-major order: the SMs work on the same one or two chunks at
        // any time, which keeps their maps and bricks in L1 / L2) -- no election, no block-level barrier, no tail behind a
        // chunk switch.
        if (!kSmemMaps && !first_chunk) break;
        if (own_next >= a.num_chunks && a.num_chunks == 1 && kSmemMaps) break;  // a single chunk: nothing to steal
        if (!first_chunk) {
            __syncthreads();  // all warps are done reading the maps before the next chunk's copy overwrites them
            if (kSmemMaps) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        int code = -1;
        if (!kSmemMaps) {
            code = 1;  // placeholder chunk 0: the chunk follows from the tile, see bind_chunk
        } else if (own_next < a.num_chunks) {
            code = own_next * 2 + 1;  // (every thread knows: no election)
        } else {
            if (warp == 0) {
                // candidates (blockIdx + k) % B, k = steal_k + 1 ..., 32 at a time: every lane looks at one counter
                int pick = -1;
                while (pick < 0 && steal_k + 1 < a.num_chunks) {
                    const int k = steal_k + 1 + lane;
                    bool open = false;
                    int cand = 0;
                    if (k < a.num_chunks) {
                        cand = (int)((blockIdx.x + (unsigned)k) % (unsigned)a.num_chunks);
                        const int owners = cand < (int)gridDim.x ? ((int)gridDim.x - 1 - cand) / a.num_chunks + 1 : 1;
                        const int fixed = min(total_tiles, owners * kWarps);  // tiles dealt statically to the chunk's owners
                        open = fixed + *reinterpret_cast<volatile int32_t *>(a.tile_counter + cand) < total_tiles;
                    }
                    const unsigned m = __ballot_sync(kFull, open);
                    if (m) {
                        const int src = __ffs(m) - 1;
                        pick = __shfl_sync(kFull, cand, src) * 2;
                        steal_k += src + 1;
                    } else {
                        steal_k += 32;
                    }
                }
                if (lane == 0) s_next_chunk = pick;
            }
            __syncthreads();
            code = s_next_chunk;
        }
        if (code < 0) break;
        int chunk = code >> 1;
        const bool own = (code & 1) != 0;
        if (own) own_next += (int)gridDim.x;
        if (kSmemMaps) {
            if (threadIdx.x == 0) {  // cell classes + block map: TMA bulk copies, completion on the mbarrier
                const unsigned vb_bytes = (unsigned)(a.vpc * sizeof(uint2)), bm_bytes = (unsigned)a.bpc;
                mbar_expect_tx(mbar, vb_bytes + bm_bytes);
                const uint8_t *src = reinterpret_cast<const uint8_t *>(a.vbits + (size_t)chunk * a.vpc);
                uint8_t *dst = reinterpret_cast<uint8_t *>(s_vbits);
                for (unsigned o = 0; o < vb_bytes; o += 32768u) bulk_copy_g2s(dst + o, src + o, min(32768u, vb_bytes - o), mbar);
                bulk_copy_g2s(s_bmap, a.bmap + (size_t)chunk * a.bpc, bm_bytes, mbar);
            }
        }
        const uint2 *vbits = kSmemMaps ? s_vbits : a.vbits + (size_t)chunk * a.vpc;   // (re-bound per tile in global mode)
        const uint8_t *bmap = kSmemMaps ? s_bmap : a.bmap + (size_t)chunk * a.bpc;
        Volume v;
        v.index = a.sparse_mapping;
        v.sdf = a.vals_sdf;
        v.dense = a.dense;
        v.cell0 = (unsigned)chunk * (unsigned)cells;
        v.dimx = a.dimx; v.dimy = a.dimy; v.dimz = a.dimz;
        v.guard = a.guard;

        // CTAs that share this chunk: ranks 0..group-1.  First round static and contiguous per CTA, then dynamic.
        const int nb = a.num_chunks;
        const int group = chunk < (int)gridDim.x ? ((int)gridDim.x - 1 - chunk) / nb + 1 : 1, rank = blockIdx.x / nb;
        // (global mode: no static round, `tile` runs over the tiles of all chunks)
        const int tile_limit = kSmemMaps ? total_tiles : total_tiles * nb;
        const int static_tiles = kSmemMaps ? min(total_tiles, group * kWarps) : 0;
        const int per = static_tiles / group, extra = static_tiles - per * group;
        const int my_first = rank * per + min(rank, extra), my_count = (own && kSmemMaps) ? per + (rank < extra ? 1 : 0) : 0;
        int tile = warp < my_count ? my_first + warp : tile_limit;
        int32_t *counter = a.tile_counter + (kSmemMaps ? chunk : 0);
        if (tile >= tile_limit && static_tiles < tile_limit) {
            int t = 0;
            if (lane == 0) t = static_tiles + atomicAdd(counter, 1);
            tile = __shfl_sync(kFull, t, 0);
        }
        // global mode: the chunk of a tile, its volume and maps; returns the tile's index within the chunk
        auto bind_chunk = [&](int t) -> int {
            if (kSmemMaps) return t;
            chunk = t / total_tiles;
            v.cell0 = (unsigned)chunk * (unsigned)cells;
            vbits = a.vbits + (size_t)chunk * a.vpc;
            bmap = a.bmap + (size_t)chunk * a.bpc;
            return t - chunk * total_tiles;
        };

        // Per-lane ray of the warp's current tile: set up (and clipped against the grid) before the chunk's maps are needed,
        // so that the first tile's set-up overlaps the TMA copies.
        struct TileRay {
            Ray r;
            float invx, invy, invz, kx, ky, kz;
            int sxm, sym, szm;
            float ray, t_end;
            int jump_cap;
            unsigned pix;
            size_t gpix;
            bool active, inside;
            int img, view, wx0, wy0;
#ifdef SPSG_STATS
            long long clk0;
#endif
        };
        auto prepare = [&](int tile, TileRay &q) {
            const int view = tile / tiles_per_image, tt = tile - view * tiles_per_image;
            const int blk = tt >> 2, sub = tt & 3;
            const int by = blk / blocks_x, bx = blk - by * blocks_x;
            const int wx0 = (bx * 2 + (sub & 1)) * kWarpW, wy0 = (by * 2 + (sub >> 1)) * kWarpH;
            const int img = chunk * a.views + view;
            q.view = view; q.img = img; q.wx0 = wx0; q.wy0 = wy0;
            q.inside = wx0 < a.width && wy0 < a.height;
            if (q.inside) {
                const unsigned ux = wx0 + (lane & 7), uy = wy0 + (lane >> 3);
                const bool active = ux < (unsigned)a.width && uy < (unsigned)a.height;
                const unsigned pix = uy * a.width + ux;
                const size_t gpix = (size_t)img * a.width * a.height + pix;

#ifdef SPSG_STATS
                q.clk0 = clock64();
#endif
                // Lanes outside the image run the same loops below with an exhausted ray.
                const Ray r = setup_ray(a.view_matrix + (size_t)img * 16, a.intrinsics + (size_t)img * 4,
                                        active ? ux : 0u, active ? uy : 0u, a.depth_min, a.depth_max);
                // approximate reciprocals are only used to size jumps; every margin below dwarfs their error
                const float invx = r.dx != 0.0f ? rcp_approx(r.dx) : 0.0f, invy = r.dy != 0.0f ? rcp_approx(r.dy) : 0.0f,
                            invz = r.dz != 0.0f ? rcp_approx(r.dz) : 0.0f;
                // exit-plane constants of the region jumps: t = (face -+ kBoxEps - cam) / dir, +inf for an axis-parallel ray
                const float kx = r.dx != 0.0f ? ((r.dx > 0.0f ? -kBoxEps : kBoxEps) - r.camx) * invx : kInf;
                const float ky = r.dy != 0.0f ? ((r.dy > 0.0f ? -kBoxEps : kBoxEps) - r.camy) * invy : kInf;
                const float kz = r.dz != 0.0f ? ((r.dz > 0.0f ? -kBoxEps : kBoxEps) - r.camz) * invz : kInf;
                const int sxm = r.dx > 0.0f ? -1 : 0, sym = r.dy > 0.0f ? -1 : 0, szm = r.dz > 0.0f ? -1 : 0;
                float ray = r.t0, t_end = active ? r.t1 : -kInf;
                // A closed-form jump of j steps lands within j * ulp(ray) / 2 of ray + j * inc (step_advance): cap j so that
                // this drift stays below kBoxEps / 4, far inside the kBoxEps the skip regions are shrunk by.
                int jump_cap = 1 << 22;
                {
                    const float top = fmaxf(fabsf(r.t1), 1.0f);
                    const float ulp = __uint_as_float(__float_as_uint(top) & 0x7f800000u) * 1.1920928955078125e-07f;
                    const float cap = (0.5f * kBoxEps) / ulp;
                    jump_cap = cap < 4194304.0f ? max(1, __float2int_rd(cap)) : (1 << 22);
                }
                if (clip && active) {
                    // Samples are valid only for p in (0, dim-1) on every axis (all 8 corners inside the grid).
                    float tin = -kInf, tout = kInf;
#define SPSG_SLAB(o, d, inv, lo, hi)                                        \
    if ((d) != 0.0f) {                                                      \
        const float ta_ = ((lo) - (o)) * (inv), tb_ = ((hi) - (o)) * (inv); \
        tin = fmaxf(tin, fminf(ta_, tb_));                                  \
        tout = fminf(tout, fmaxf(ta_, tb_));                                \
    } else if ((o) < (lo) || (o) > (hi)) {                                  \
        tin = kInf;                                                         \
        tout = -kInf;                                                       \
    }
                    SPSG_SLAB(r.camx, r.dx, invx, -kBoxEps, (float)(a.dimx - 1) + kBoxEps)
                    SPSG_SLAB(r.camy, r.dy, invy, -kBoxEps, (float)(a.dimy - 1) + kBoxEps)
                    SPSG_SLAB(r.camz, r.dz, invz, -kBoxEps, (float)(a.dimz - 1) + kBoxEps)
#undef SPSG_SLAB
                    const float margin = 0.0625f;
                    if (!(tin <= tout)) {
                        t_end = -kInf;  // misses the grid: nothing to march
                    } else {
                        t_end = fminf(t_end, tout + margin);
                        // jump to (at most) the last sample before tin - margin
                        while (ray < tin - margin - a.inc && ray < t_end) {
                            const int want = max(1, min(__float2int_rd((tin - margin - ray) * inv_inc) - 1, jump_cap));
                            ray = step_advance(s_steps, a.inc, ray, want);
                        }
                        // The samples between there and the first one with floor(p) in [0, dim - 1) on every axis are
                        // invalid (see the march) and the march state is still "no valid sample": step over them here,
                        // one real add each, instead of spending a warp iteration on each of them.
                        for (int k = 0; k < 6 && ray < t_end; k++) {
                            const int ix = __float2int_rd(__fmaf_rn(r.dx, ray, r.camx)), iy = __float2int_rd(__fmaf_rn(r.dy, ray, r.camy)),
                                      iz = __float2int_rd(__fmaf_rn(r.dz, ray, r.camz));
                            if ((unsigned)ix < (unsigned)a.vx && (unsigned)iy < (unsigned)a.vy && (unsigned)iz < (unsigned)a.vz) break;
                            if (!skip_ok) break;
                            ray = __fadd_rn(ray, a.inc);
                        }
                    }
                }
                q.r = r; q.invx = invx; q.invy = invy; q.invz = invz; q.kx = kx; q.ky = ky; q.kz = kz;
                q.sxm = sxm; q.sym = sym; q.szm = szm; q.ray = ray; q.t_end = t_end; q.jump_cap = jump_cap;
                q.pix = pix; q.gpix = gpix; q.active = active;
            }
        };
        TileRay q;
        q.inside = false;
        if (tile < tile_limit) prepare(bind_chunk(tile), q);
        if (kSmemMaps) mbar_wait(mbar, phase);  // the chunk's class planes and block map have landed

        while (tile < tile_limit) {
            int next = tile_limit;
            if (lane == 0 && static_tiles < tile_limit) next = static_tiles + atomicAdd(counter, 1);  // prefetched
            if (q.inside) {
                const Ray r = q.r;
                const float invx = q.invx, invy = q.invy, invz = q.invz, kx = q.kx, ky = q.ky, kz = q.kz;
                const int sxm = q.sxm, sym = q.sym, szm = q.szm, jump_cap = q.jump_cap;
                float ray = q.ray;
                const float t_end = q.t_end;
                const unsigned pix = q.pix;
                const size_t gpix = q.gpix;
                const bool active = q.active;
                const int img = q.img, view = q.view, wx0 = q.wx0, wy0 = q.wy0;
                int hit = -1;
                float depth = 0.0f;
#ifdef SPSG_STATS
                const long long clk0 = q.clk0;
                long long clk_march = 0, clk_refine = 0;
                int my_iters = 0;
                const long long clk1 = clock64(), clk1b = clk1;
#endif

                // last valid sample (kernel.cu:64-69).  "No valid last sample" is encoded as last_sdf == 0: a last value of
                // +-0 can never satisfy the strict sign test (:205) either, so the two are indistinguishable.
                // last_lazy: last_sdf is only a +-1 placeholder carrying the sign the cell class guarantees; the value
                // is computed if and when a crossing needs it.
                float last_sdf = 0.0f, last_alpha = 0.0f;
                bool last_lazy = false;
                float dist = 0.0f;
                enum { kMarch = 0, kCross = 1, kDone = 2 };
                int state = kMarch;

                for (;;) {
#ifdef SPSG_STATS
                    const long long clk_a = clock64();
#endif
                    // ---- march.  The loop is warp-synchronous: all lanes take part in every vote and every iteration
                    // handles one event per marching lane, so diverged lanes re-join at the bottom of each iteration
                    // instead of running their iterations one group after the other.  An event is either a jump over
                    // samples whose outcome is known from the block map, or one sample.
                    while (__any_sync(kFull, state == kMarch)) {
#ifdef SPSG_STATS
                        my_iters++;
                        if (lane == 0) EVT_ADD(8, 1);
                        { const int nm = __popc(__ballot_sync(kFull, state == kMarch)); if (lane == 0) EVT_ADD(14, nm); }
#endif
                        if (state == kMarch) {
                            if (!(ray < t_end)) {  // kernel.cu:200
                                state = kDone;
                            } else {
                                enum { kActExact = 0, kActDense = 1, kActInvalid = 2, kActSign = 3, kActJumpEmpty = 4, kActJumpSame = 5 };
                                int act = kActExact, nadv = 1;
                                float sgn = 0.0f, wx = 0.0f, wy = 0.0f, wz = 0.0f;
                                const float px = __fmaf_rn(r.dx, ray, r.camx), py = __fmaf_rn(r.dy, ray, r.camy),
                                            pz = __fmaf_rn(r.dz, ray, r.camz);
                                // floor: one conversion on the address path (exact for every in-grid p; an out-of-range p
                                // saturates and fails the bounds test below)
                                const int ix = __float2int_rd(px), iy = __float2int_rd(py), iz = __float2int_rd(pz);
                                const float fx = (float)ix, fy = (float)iy, fz = (float)iz;
                                if ((unsigned)ix < (unsigned)a.vx && (unsigned)iy < (unsigned)a.vy && (unsigned)iz < (unsigned)a.vz) {
                                    // block map and cell class are fetched together (independent shared-memory addresses)
                                    const int b = bmap[((iz >> kFineLog2) * a.nby + (iy >> kFineLog2)) * a.nbx + (ix >> kFineLog2)];
                                    const uint2 word = vbits[(iz * a.dimy + iy) * a.wpr + (ix >> 5)];
                                    wx = __fadd_rn(px, -fx); wy = __fadd_rn(py, -fy); wz = __fadd_rn(pz, -fz);
                                    const float wlo = fminf(wx, fminf(wy, wz)), whi = fmaxf(wx, fmaxf(wy, wz));
                                    if (b != 0 && wlo >= kBoxEps && whi <= 1.0f - kBoxEps) {
                                        // p is inside an aligned uniform region of edge `size`, at least kBoxEps away from
                                        // every cell face and hence from the region's faces: corner (0,0,0) of this sample
                                        // and of every later one up to the region's (shrunk) exit lies in the region.
                                        const int kind = b >> 3, size = 2 << (b & 7), mask = ~(size - 1);
                                        // a sign-uniform region cannot be jumped while the last valid sample has the
                                        // other sign: its first valid sample would be a crossing
                                        const bool opposite = (kind == kKindPos && last_sdf < 0.0f) ||
                                                              (kind == kKindNeg && last_sdf > 0.0f);
                                        if (!opposite) {
                                            // exit face per axis = origin + (dir > 0 ? size : 0), shrunk by kBoxEps (folded
                                            // into kx/ky/kz together with the camera position)
                                            const float tx_ = __fmaf_rn((float)((ix & mask) + (size & sxm)), invx, kx);
                                            const float ty_ = __fmaf_rn((float)((iy & mask) + (size & sym)), invy, ky);
                                            const float tz_ = __fmaf_rn((float)((iz & mask) + (size & szm)), invz, kz);
                                            const float tout = fminf(tx_, fminf(ty_, tz_));
                                            // steps to the first sample beyond the region's exit
                                            const int n = max(1, min(__float2int_rd((tout - ray) * inv_inc) + 1, jump_cap));
                                            if (kind == kKindEmpty) {
                                                // every sample before that one is invalid (kernel.cu:131,259)
                                                act = kActJumpEmpty; nadv = n;
                                            } else if (n >= 2) {
                                                // Samples up to the last one inside are invalid or share the region's sign,
                                                // and so does the last valid one before them: no crossing.  Land on the
                                                // last one inside; it is classified by its own cell and leaves the march
                                                // state exactly as the reference's sample-by-sample walk would.
                                                act = kActJumpSame; nadv = n - 1;
                                            }
                                        }
                                    }
                                    if (act == kActExact) {
                                        // One sample, decided by its own cell.  With frac(p) clear of the cell faces the
                                        // reference's corners are exactly floor(p) + {0,1}; the cell's class says whether
                                        // all 8 are present and whether they share a sign.
                                        const float g = frac_guard(v.guard, ix, iy, iz);
                                        if (wlo >= g && whi <= 1.0f - g) {
                                            const unsigned ca = (word.x >> (ix & 31)) & 1u, cb = (word.y >> (ix & 31)) & 1u;
                                            if ((ca | cb) == 0u) {
                                                act = kActInvalid;
                                            } else {
                                                act = kActDense;
                                                if ((ca & cb) == 0u) {
                                                    sgn = ca ? 1.0f : -1.0f;
                                                    // opposite strict signs <=> last_sdf * (+-1) < 0 (last_sdf is never NaN)
                                                    if (!(__fmul_rn(last_sdf, sgn) < 0.0f)) act = kActSign;
                                                }
                                            }
                                        }
                                    }
                                } else if (skip_ok) {
                                    // p < 0 or p >= dim - 1 on some axis: corner 0 rounds to -1 (p - 0.5 <= -0.5 rounds away
                                    // from zero) or corner 1 to >= dim (p - 0.5, + 1 and + 0.5 are monotonic and exact at
                                    // dim - 1), so the reference's bounds test (:131) fails -- an invalid sample, no arithmetic.
                                    // (NaN coordinates convert to 0 and never get here.)
                                    act = kActInvalid;
                                }
                                EVT_ADD(act, 1); EVT_ADD(9, 1); EVT_ADD(10, nadv);
                                if (act <= kActDense) {
                                    if (act == kActDense) {
                                        dist = sample_dense(v, ix, iy, iz, wx, wy, wz);
                                    } else {
                                        dist = sample_sdf(v, fast_ok, px, py, pz);  // the reference's exact corner arithmetic
                                    }
                                    const bool valid = dist == dist;
                                    if (valid && ((last_sdf > 0.0f && dist < 0.0f) || (last_sdf < 0.0f && dist > 0.0f))) {  // :205
                                        state = kCross;
                                    } else {
                                        last_sdf = valid ? dist : 0.0f; last_alpha = ray; last_lazy = false;  // :254-256 / :259
                                    }
                                } else if (act == kActSign) {
                                    last_sdf = sgn; last_alpha = ray; last_lazy = true;  // :254-256
                                } else if (act != kActJumpSame) {
                                    last_sdf = 0.0f;  // :259 (invalid sample, or a run of them)
                                }
                                if (state == kMarch) ray = step_advance(s_steps, a.inc, ray, nadv);  // :257,:260
                            }
                        }
                    }
#ifdef SPSG_STATS
                    const long long clk_b = clock64();
                    clk_march += clk_b - clk_a;
#endif
                    // ---- refinement round: every lane is either waiting with a crossing or finished
                    if (!__any_sync(kFull, state == kCross)) break;
                    if (lane == 0) EVT_ADD(11, 1);
                    if (state == kCross) {
                        EVT_ADD(12, 1);
                        if (last_lazy) {  // the crossing needs the previous sample's value after all (its class says it is valid)
                            const float dl = sample_sdf(v, fast_ok, __fmaf_rn(r.dx, last_alpha, r.camx),
                                                        __fmaf_rn(r.dy, last_alpha, r.camy), __fmaf_rn(r.dz, last_alpha, r.camz));
                            if (dl == dl) last_sdf = dl;
                            last_lazy = false;
                        }
                        // findIntersectionBisection (:166-187)
                        float ta = last_alpha, da = last_sdf, tb = ray, db = dist, c = 0.0f;
                        float cx = 0.0f, cy = 0.0f, cz = 0.0f;
                        bool ok = true;
#pragma unroll 1
                        for (int k = 0; k < 3; k++) {
                            c = __fmaf_rn(__fadd_rn(tb, -ta), __fdiv_rn(da, __fadd_rn(da, -db)), ta);  // :161
                            cx = __fmaf_rn(r.dx, c, r.camx);
                            cy = __fmaf_rn(r.dy, c, r.camy);
                            cz = __fmaf_rn(r.dz, c, r.camz);
                            const float dc = sample_sdf(v, fast_ok, cx, cy, cz);
                            if (dc != dc) {
                                ok = false;
                                break;
                            }
                            if (__fmul_rn(da, dc) > 0.0f) { ta = c; da = dc; } else { tb = c; db = dc; }  // :180-181
                        }
                        if (ok && fabsf(__fadd_rn(last_sdf, -dist)) < a.thresh && fabsf(dist) < a.thresh) {  // :211-213
                            depth = __fdiv_rn(c, r.d2r);                                                     // :215
                            // payload voxel = nearest voxel of the last refinement point (:129) == hit voxel
                            // round(cam + alpha*dir) (:241-242, same fma).  It is one of the 8 present corners; if rounding
                            // ever says otherwise the reference reads stale registers -- we keep marching instead.
                            const int nx = round_voxel(cx), ny = round_voxel(cy), nz = round_voxel(cz);
                            hit = in_grid(v, nx, ny, nz) ? __ldg(v.index + (v.cell0 + (unsigned)((nz * v.dimy + ny) * v.dimx + nx))) : -1;
                        }
                        if (hit >= 0) {
                            state = kDone;
                        } else {
                            last_sdf = dist; last_alpha = ray; last_lazy = false;  // :254-256
                            ray = __fadd_rn(ray, a.inc);                           // :257
                            state = kMarch;
                        }
                    }
#ifdef SPSG_STATS
                    clk_refine += clock64() - clk_b;
#endif
                }
#ifdef SPSG_STATS
                const long long clk2 = clock64();
#endif

                if (kLabels) {
                    // ---- label epilogue: one byte per pixel (a tile row is 8 contiguous bytes), one shared atomic per
                    // distinct label of the warp
                    const int C = a.loss.sem_channels;
                    const int label = hit >= 0 ? min((int)__ldg(a.voxel_labels + hit), C) : C;
                    if (active) a.image_label[gpix] = (uint8_t)label;
                    if (a.hist) {
                        const unsigned peers = __match_any_sync(kFull, active ? label : -1);
                        if (active && lane == __ffs(peers) - 1)
                            atomicAdd(reinterpret_cast<unsigned *>(smem + 128) + label, (unsigned)__popc(peers));
                    }
                } else if (kEval) {
                    // ---- eval epilogue: predicted label, confusion count (one shared atomic per distinct cell of the
                    // warp), the loss terms of kLoss from the hit voxel's payload rows
                    const LossArgs &L = a.loss;
                    const int C = L.sem_channels;
                    const int label = hit >= 0 ? min((int)__ldg(a.voxel_labels + hit), C) : C;
                    if (a.image_label && active) a.image_label[gpix] = (uint8_t)label;
                    if (a.confusion) {
                        const int cell = active ? min((int)L.target_label[gpix], C) * (C + 1) + label : -1;
                        const unsigned peers = __match_any_sync(kFull, cell);
                        if (active && lane == __ffs(peers) - 1)
                            atomicAdd(reinterpret_cast<unsigned *>(smem + 128) + cell, (unsigned)__popc(peers));
                    }
                    float acc[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
                    if (hit >= 0) {
                        if (L.target_depth) {  // train.py:635-638
                            const float t = __ldg(L.target_depth + gpix);
                            if (t != 0.0f) { acc[0] = fabsf(__fmul_rn(depth, L.voxelsize) - t); acc[1] = 1.0f; }
                        }
                        if (L.target_color) {  // loss.py:246-257
                            const float *c = a.vals_color + (size_t)hit * 3;
                            const float w = L.weight_color ? __ldg(L.weight_color + gpix) : 1.0f;
                            const float *t = L.target_color + gpix * 3;
                            acc[2] = fabsf(__fadd_rn(__fmul_rn(__ldg(c + 0), w), -__fmul_rn(__ldg(t + 0), w))) +
                                     fabsf(__fadd_rn(__fmul_rn(__ldg(c + 1), w), -__fmul_rn(__ldg(t + 1), w))) +
                                     fabsf(__fadd_rn(__fmul_rn(__ldg(c + 2), w), -__fmul_rn(__ldg(t + 2), w)));
                            acc[3] = 3.0f;
                        }
                        if (L.target_label) {  // train.py:744-746, over the hit voxel's C logits
                            const int y = L.target_label[gpix];
                            const float *lg = a.vals_semantic + (size_t)hit * C;
                            if (y < C && __ldg(lg) != -kInf) {
                                const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
                                acc[4] = w * ce_nll<true>(lg, C, y);
                                acc[5] = w;
                            }
                        }
                    }
                    // the partials exactly as kLoss forms them, stored instead of added
                    float mine = 0.0f;
                    const int n_depth = __popc(__ballot_sync(kFull, acc[1] != 0.0f)), n_color = __popc(__ballot_sync(kFull, acc[3] != 0.0f));
                    if (lane == 1) mine = (float)n_depth;
                    if (lane == 3) mine = 3.0f * (float)n_color;
#pragma unroll
                    for (int k = 0; k < 6; k++) {
                        if (k == 1 || k == 3) continue;
                        const float t = warp_sum(acc[k]);
                        if (lane == k) mine = t;
                    }
                    if (lane < 6) a.eval_tiles[((size_t)img * tiles_per_image + tile % tiles_per_image) * 8 + lane] = mine;
                } else {
                // ---- write-out (kernel.cu:276-285 init, :217-239 hit) through shared memory
                const float ninf = __int_as_float(0xff800000);
                float col0 = ninf, col1 = ninf, col2 = ninf, dep = ninf;
                float sem[14];
#pragma unroll
                for (int k = 0; k < 14; k++) sem[k] = ninf;
                float n0 = ninf, n1 = ninf, n2 = ninf;
                bool first = false;
                if (hit >= 0) {
                    const float *c = a.vals_color + (size_t)hit * 3;
                    const float *n = a.vals_normal + (kViewNormals ? ((size_t)hit * a.views + view) * 3 : (size_t)hit * 3);
                    col0 = __ldg(c + 0); col1 = __ldg(c + 1); col2 = __ldg(c + 2);
                    const float m0 = __ldg(n + 0), m1 = __ldg(n + 1), m2 = __ldg(n + 2);
                    if (!(m0 == 0.0f && m1 == 0.0f && m2 == 0.0f)) { n0 = m0; n1 = m1; n2 = m2; }  // :220
                    dep = depth;
                    if (!kGenericSem) {
                    const float2 *s2 = reinterpret_cast<const float2 *>(a.vals_semantic + (size_t)hit * 14);
#pragma unroll
                    for (int k = 0; k < 7; k++) {
                        const float2 t2 = __ldg(s2 + k);
                        sem[2 * k] = t2.x; sem[2 * k + 1] = t2.y;
                    }
                    }
                }
                {
                    // voxel -> pixel registration (:244-247), one atomic per distinct voxel of the warp: lanes that hit
                    // the same voxel take consecutive slots from a single atomicAdd (the reference's slot order is the
                    // arbitrary order of its per-pixel atomics)
                    const unsigned peers = __match_any_sync(kFull, hit);
                    if (hit >= 0) {
                        const int leader = __ffs(peers) - 1;
                        const size_t row = (size_t)view * (size_t)a.num_locs + (size_t)hit;
                        int base = 0;
                        if (lane == leader) base = atomicAdd(a.mapping3dto2d_num + row, __popc(peers));
                        base = __shfl_sync(peers, base, leader);
                        const int offset = base + __popc(peers & ((1u << lane) - 1));
                        if (offset < a.max_pixels) a.mapping3dto2d[row * a.max_pixels + offset] = (int)pix;
                        first = offset == 0;
                    }
                }
#ifdef SPSG_STATS
                // force the payload + atomic results before reading the clock
                const long long clk_e1 = (col0 != 12345.0f && sem[13] != 12345.0f && !(first && dep == 54321.0f)) ? clock64() : 0;
#endif
                // the first pixel of a (voxel, view) pair appends the pair to the backward's work list: one atomic per
                // warp, issued here and consumed after the image stores so that its round trip overlaps them
                const unsigned list_mask = __ballot_sync(kFull, first);
                int list_base = 0;
#ifndef SPSG_NO_LIST
                if (list_mask && lane == 0) list_base = atomicAdd(a.list_count, __popc(list_mask));
#endif
                if (a.hits && active) a.hits[gpix] = hit;
#ifdef SPSG_STATS
                const long long clk_e2 = clock64();
#endif

                // the staging buffer is reused: semantic first, then colour + normal + depth
                const bool vec = a.vec_ok != 0;
                const size_t tile_pix0 = ((size_t)img * a.height + wy0) * a.width + wx0;
                if (kGenericSem) {
                    store_semantic_rows(a.vals_semantic, a.loss.sem_channels, hit, a.image_semantic, tile_pix0, wx0, wy0, a.width,
                                        a.height, lane);
                } else {
#pragma unroll
                for (int k = 0; k < 7; k++) reinterpret_cast<float2 *>(stage + lane * 14)[k] = make_float2(sem[2 * k], sem[2 * k + 1]);
                __syncwarp();
                store_warp_tile<14>(stage, a.image_semantic, tile_pix0, wx0, wy0, a.width, a.height, vec, lane);
                }
                if (kLoss) {
                    // The three 2D loss terms of this pixel.  The logits are read back from the staging row (still intact: the
                    // stores above only read it), one at a time, so the 14 payload registers are dead by now and the fused
                    // variant needs no more registers than the plain one.
                    float acc[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
                    if (hit >= 0) {
                        const LossArgs &L = a.loss;
                        if (L.target_depth) {  // train.py:635-638
                            const float t = __ldg(L.target_depth + gpix);
                            if (t != 0.0f) { acc[0] = fabsf(__fmul_rn(depth, L.voxelsize) - t); acc[1] = 1.0f; }
                        }
                        if (L.target_color) {  // loss.py:246-257
                            const float w = L.weight_color ? __ldg(L.weight_color + gpix) : 1.0f;
                            const float *t = L.target_color + gpix * 3;
                            acc[2] = fabsf(__fadd_rn(__fmul_rn(col0, w), -__fmul_rn(__ldg(t + 0), w))) +
                                     fabsf(__fadd_rn(__fmul_rn(col1, w), -__fmul_rn(__ldg(t + 1), w))) +
                                     fabsf(__fadd_rn(__fmul_rn(col2, w), -__fmul_rn(__ldg(t + 2), w)));
                            acc[3] = 3.0f;
                        }
                        if (kGenericSem && L.target_label) {  // the same over the hit voxel's C logits
                            const int y = L.target_label[gpix];
                            const int C = a.loss.sem_channels;
                            const float *lg = a.vals_semantic + (size_t)hit * C;
                            if (y < C && __ldg(lg) != ninf) {
                                const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
                                acc[4] = w * ce_nll<true>(lg, C, y);
                                acc[5] = w;
                            }
                        } else if (L.target_label) {  // train.py:744-746
                            const int y = L.target_label[gpix];
                            const float *lg = stage + lane * 14;
                            if (y < 14 && lg[0] != ninf) {  // valid = (label < 14) & (logit0 != -inf), train.py:744
                                float m = lg[0];
#pragma unroll
                                for (int k = 1; k < 14; k++) m = fmaxf(m, lg[k]);
                                float s = 0.0f;
#pragma unroll
                                for (int k = 0; k < 14; k++) s += __expf(lg[k] - m);  // arguments <= 0, the largest term is exactly 1:
                                // relative error of the sum <= 2^-21, of the loss far below the 1e-5 it is checked to
                                const float w = L.class_weight ? __ldg(L.class_weight + y) : 1.0f;
                                acc[4] = w * (__logf(s) + m - lg[y]);
                                acc[5] = w;
                            }
                        }
                    }
                    // the two pixel counts are ballots, the four sums shuffle trees
                    float mine = 0.0f;
                    const int n_depth = __popc(__ballot_sync(kFull, acc[1] != 0.0f)), n_color = __popc(__ballot_sync(kFull, acc[3] != 0.0f));
                    if (lane == 1) mine = (float)n_depth;
                    if (lane == 3) mine = 3.0f * (float)n_color;
#pragma unroll
                    for (int k = 0; k < 6; k++) {
                        if (k == 1 || k == 3) continue;
                        const float t = warp_sum(acc[k]);
                        if (lane == k) mine = t;
                    }
                    // one double atomic per warp and term, spread over kLossSlots copies of the accumulators
                    const unsigned slot = ((unsigned)tile * 7u + (unsigned)img * 11u) % kLossSlots;
                    if (lane < 6 && mine != 0.0f) atomicAdd(a.loss.accum + slot * 8 + lane, (double)mine);
                }
                __syncwarp();
                float *s_col = stage, *s_nrm = stage + 96, *s_dep = stage + 192;
                s_col[lane * 3 + 0] = col0; s_col[lane * 3 + 1] = col1; s_col[lane * 3 + 2] = col2;
                s_nrm[lane * 3 + 0] = n0; s_nrm[lane * 3 + 1] = n1; s_nrm[lane * 3 + 2] = n2;
                s_dep[lane] = dep;
                __syncwarp();
                store_warp_tile<3>(s_col, a.image_color, tile_pix0, wx0, wy0, a.width, a.height, vec, lane);
                store_warp_tile<3>(s_nrm, a.image_normal, tile_pix0, wx0, wy0, a.width, a.height, vec, lane);
                store_warp_tile<1>(s_dep, a.image_depth, tile_pix0, wx0, wy0, a.width, a.height, vec, lane);
                __syncwarp();
#ifndef SPSG_NO_LIST
                if (list_mask) {
                    list_base = __shfl_sync(kFull, list_base, 0);
                    if (first) a.list[list_base + __popc(list_mask & ((1u << lane) - 1))] = make_int2(hit, img);
                }
#endif
#ifdef SPSG_STATS
                if (lane == 0) {
                    const long long clk3 = clock64();
                    STAT_ADD(16, clk1 - clk0); STAT_MAX(17, clk1 - clk0);        // setup + clip
                    STAT_ADD(28, clk1b - clk1); STAT_MAX(29, clk1b - clk1);      // wait for the maps
                    STAT_ADD(18, clk_march); STAT_MAX(19, clk_march);            // march
                    STAT_ADD(20, clk_refine); STAT_MAX(21, clk_refine);          // refinement
                    STAT_ADD(22, clk3 - clk2); STAT_MAX(23, clk3 - clk2);        // epilogue
                    STAT_ADD(40, clk_e1 - clk2); STAT_MAX(41, clk_e1 - clk2);    // payload + registration atomics
                    STAT_ADD(42, clk_e2 - clk_e1); STAT_MAX(43, clk_e2 - clk_e1);  // list append
                    STAT_ADD(44, clk3 - clk_e2); STAT_MAX(45, clk3 - clk_e2);    // staging + stores
                    STAT_ADD(24, clk3 - clk0); STAT_MAX(25, clk3 - clk0);        // whole tile
                    STAT_MAX(26, my_iters);
                    if (tile < 131072) {
                        unsigned smid;
                        asm("mov.u32 %0, %%smid;" : "=r"(smid));
                        int *ts = g_tile_stats[tile];
                        ts[0] = (int)(clk3 - clk0); ts[1] = (int)(clk1 - clk0); ts[2] = (int)clk_march; ts[3] = (int)clk_refine;
                        ts[4] = (int)(clk3 - clk2); ts[5] = my_iters; ts[6] = (int)smid; ts[7] = (int)(clk0 & 0x7fffffff);
                    }
                    STAT_ADD(27, my_iters);
                    int bucket = 0;
                    for (int t = my_iters; t > 8; t >>= 1) bucket++;
                    STAT_ADD(32 + min(bucket, 9), 1);
                }
#endif
                }  // !kLabels && !kEval
            } else if (kEval && lane < 6) {
                a.eval_tiles[((size_t)q.img * tiles_per_image + tile % tiles_per_image) * 8 + lane] = 0.0f;  // no pixel
            }
            tile = __shfl_sync(kFull, next, 0);
            if (tile < tile_limit) prepare(bind_chunk(tile), q);
        }
        if (kSmemMaps) phase ^= 1u;
    }
    if (kLabels && a.hist) {
        __syncthreads();
        const unsigned *s_hist = reinterpret_cast<const unsigned *>(smem + 128);
        if (threadIdx.x <= a.loss.sem_channels && s_hist[threadIdx.x])
            atomicAdd(a.hist + threadIdx.x, (unsigned long long)s_hist[threadIdx.x]);
    }
    if (kEval && a.confusion) {
        __syncthreads();
        const unsigned *s_conf = reinterpret_cast<const unsigned *>(smem + 128);
        for (int i = threadIdx.x; i < conf_cells; i += kWarps * 32)
            if (s_conf[i]) atomicAdd(a.confusion + i, (unsigned long long)s_conf[i]);
    }
    if (kLoss) {
        // Every loss atomic of this CTA is ordered before its arrival; the CTA that arrives last sees them all in L2 and
        // forms the means and the total (what a separate one-warp launch did: 4 us of a 57 us C2 step).
        __shared__ int s_last;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            s_last = atomicAdd(a.loss.done, 1) == (int)gridDim.x - 1;
        }
        __syncthreads();
        if (s_last && warp == 0) {
            __threadfence();
            finalize_loss_warp(a.loss.accum, a.loss.loss_out, a.loss.w_depth, a.loss.w_color, a.loss.w_sem,
                               a.loss.target_depth != nullptr, a.loss.target_color != nullptr, a.loss.target_label != nullptr, lane);
        }
    }
}


// loss_out[0..3] = depth, colour, semantic, weighted total; [4..6] = normalisers the backward needs.
// One warp: lane l sums slots l, l + 32, ...; xor-shuffle tree over the lanes (fixed order: deterministic).
__device__ __forceinline__ void finalize_loss_warp(const double *acc, float *__restrict__ out, float w_depth, float w_color,
                                                   float w_sem, bool has_depth, bool has_color, bool has_sem, int lane) {
    double t[6] = {0, 0, 0, 0, 0, 0};
    for (int s = lane; s < kLossSlots; s += 32)
#pragma unroll
        for (int k = 0; k < 6; k++) t[k] += __ldcg(acc + s * 8 + k);  // (L2: other CTAs' atomics, see the forward kernel)
#pragma unroll
    for (int k = 0; k < 6; k++)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t[k] += __shfl_xor_sync(0xffffffffu, t[k], o);
    if (lane == 0) {
        const float ld = has_depth ? (float)(t[0] / t[1]) : 0.0f;  // mean over an empty set is NaN, like torch.mean
        const float lc = has_color ? (float)(t[2] / t[3]) : 0.0f;
        const float ls = has_sem ? (float)(t[4] / t[5]) : 0.0f;
        out[0] = ld; out[1] = lc; out[2] = ls;
        out[3] = w_depth * ld + w_color * lc + w_sem * ls;
        out[4] = (float)t[1]; out[5] = (float)t[3]; out[6] = (float)t[5];
        out[7] = 0.0f;
    }
}

__global__ void __launch_bounds__(32) finalize_loss_kernel(const double *__restrict__ acc, float *__restrict__ out,
                                                           float w_depth, float w_color, float w_sem, int has_depth,
                                                           int has_color, int has_sem) {
    finalize_loss_warp(acc, out, w_depth, w_color, w_sem, has_depth != 0, has_color != 0, has_sem != 0, threadIdx.x);
}
