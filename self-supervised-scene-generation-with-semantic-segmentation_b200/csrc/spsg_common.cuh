// spsg_common.cuh -- constants, error plumbing, kernel timing hooks, workspace layout.
// Fragment of libspsg_raycast.so: included by spsg_raycast.cu INSIDE its anonymous namespace, in the order listed there
// (one translation unit; every device function is inlined into the kernels that use it).
#pragma once

constexpr int kFineLog2 = 2;             // finest region: 4^3 voxels ("block")
constexpr int kFine = 1 << kFineLog2;
constexpr int kSuper = 8;                // hierarchy kernel handles 8^3 blocks = 32^3 voxels per CTA
constexpr float kBoxEps = 1.0f / 64.0f;  // shrink of skip regions; >> every fp32 error term (DESIGN.md)
constexpr float kFracGuard = 1.0f / 256.0f;  // fast corner path needs frac(p) in [guard, 1-guard]
constexpr int kMaxFastDim = 8192;        // fast corner path proven for coordinates < 2^13
constexpr int kLossSlots = 64;           // copies of the loss accumulators (spreads atomic contention)
constexpr int kMaxSemanticChannels = 64; // largest C of spsg_raycast_params.semantic_channels

// block map byte = kind << 3 | level; level k >= 1: the aligned region of edge 2^(k+1) voxels around the block
enum { kKindSurface = 0, kKindEmpty = 1, kKindPos = 2, kKindNeg = 3 };

thread_local char g_err[512] = "";

int fail(int code, const char *msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}
int fail_cuda(cudaError_t e, const char *where) {
    snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
    return SPSG_ERR_CUDA;
}
#define CUDA_TRY(x)                                      \
    do {                                                 \
        cudaError_t e_ = (x);                            \
        if (e_ != cudaSuccess) return fail_cuda(e_, #x); \
    } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

constexpr int kDetLossPix = 4096;  // pixels per partial of the deterministic loss sums (spsg_deterministic.cuh)
constexpr int kSegWarpSort = 64;   // SPSG_FLAG_ALL_PIXELS + DETERMINISTIC: longest segment one warp sorts (spsg_segments.cuh)
inline size_t det_loss_partials_bytes(long long num_pixels) {
    return align_up((size_t)((num_pixels + kDetLossPix - 1) / kDetLossPix) * 8 * sizeof(double), 256);
}

// Optional per-kernel timing (bench.py's roofline leg): CUDA event pairs recorded on the launch stream around the
// two dominant kernels.  Off by default; not usable during stream capture.
struct EventPair { cudaEvent_t a, b; };
bool g_timing = false;
std::vector<EventPair> g_ev[2];  // 0 = raycast_forward_kernel, 1 = backward_gather_kernel
std::mutex g_timing_mu;

struct ScopedKernelTimer {
    int which; cudaStream_t st; EventPair ev; bool on;
    ScopedKernelTimer(int w, cudaStream_t s) : which(w), st(s), on(g_timing) {
        if (on) {
            on = cudaEventCreate(&ev.a) == cudaSuccess && cudaEventCreate(&ev.b) == cudaSuccess;
            if (on) cudaEventRecord(ev.a, st);
        }
    }
    ~ScopedKernelTimer() {
        if (on) {
            cudaEventRecord(ev.b, st);
            std::lock_guard<std::mutex> lk(g_timing_mu);
            g_ev[which].push_back(ev);
        }
    }
};

// Workspace layout (caller-owned scratch, see spsg_workspace_bytes).  Written by the forward; the list, and the
// voxel->pixel tables it indexes, are what the backward of the same call pair reads.
struct Layout {
    int nbx, nby, nbz;              // 4^3 blocks per axis
    size_t bpc;                     // block-map bytes per chunk (nbx*nby*nbz rounded up to 16)
    size_t dense_off, dense_bytes;  // f32 [B][Dz][Dy][Dx], NaN = absent
    int wpr;                        // 32-cell words per x row of the cell-class bit planes
    size_t vpc;                     // uint2 words per chunk of the cell-class map (Dz*Dy*wpr rounded up to even)
    size_t vbit_off, vbit_bytes;    // uint2 [B][vpc]: bit x of (.x, .y) = class of the sample cell whose corner (0,0,0)
                                    // is the voxel: 00 invalid, 10 positive, 01 negative, 11 mixed
    size_t bmap_off, bmap_bytes;    // u8  [B][bpc] block map
    size_t marks_off, marks_bytes;  // u8  [B][bpc]: region bits of each 4^3 block (1 positive, 2 negative, 4 mixed cell)
    size_t zero_off, zero_bytes;    // everything from here to the list is cleared by the fill kernel of every forward
    size_t head_off;                // int32 list counter (256 B)
    size_t tiles_off, tiles_bytes;  // int32 [B] dynamic tile counters of the forward
    size_t arrive_off, arrive_bytes;  // int32 [B][super blocks]: classifier warps done per 32^3 super block
    size_t loss_off, loss_bytes;    // double[kLossSlots][8] loss accumulators
    size_t list_off, list_bytes;    // int2 (voxel, image) per (voxel, view) pair that received a pixel
    size_t hits_off, hits_bytes;    // optional int32 per-pixel hit voxel
    size_t det_off, det_bytes;      // SPSG_FLAG_DETERMINISTIC only: double[8] loss partials per kDetLossPix pixels
    // SPSG_FLAG_ALL_PIXELS only (else 0 bytes): the backward's per-row pixel segments (spsg_segments.cuh)
    size_t seg_head_off, seg_head_bytes;  // int32 counters: [0] segment allocator, [1] long rows
    size_t seg_end_off, seg_end_bytes;    // int32 [F*N]: end of row r's segment in the entries
    size_t seg_pix_off, seg_pix_bytes;    // int32 [B*F*W*H]: in-image pixel indices, one segment per listed row
    size_t seg_long_off, seg_long_bytes;  // with SPSG_FLAG_DETERMINISTIC: work-list items of rows longer than a warp sorts
    size_t total;
};

Layout make_layout(const spsg_raycast_params *p) {
    Layout L;
    L.nbx = (p->dimx + kFine - 1) >> kFineLog2;
    L.nby = (p->dimy + kFine - 1) >> kFineLog2;
    L.nbz = (p->dimz + kFine - 1) >> kFineLog2;
    L.bpc = align_up((size_t)L.nbx * L.nby * L.nbz, 16);
    const int F = p->views_per_chunk > 0 ? p->views_per_chunk : 1;
    const size_t cells = (size_t)p->num_chunks * p->dimz * p->dimy * p->dimx;
    size_t off = 0;
    L.dense_off = off;
    L.dense_bytes = align_up(cells * sizeof(float), 256);
    off += L.dense_bytes;
    L.wpr = (p->dimx + 31) / 32;
    L.vpc = align_up((size_t)p->dimz * p->dimy * L.wpr, 2);
    L.vbit_off = off;
    L.vbit_bytes = align_up((size_t)p->num_chunks * L.vpc * sizeof(uint2), 256);
    off += L.vbit_bytes;
    L.bmap_off = off;
    L.bmap_bytes = align_up((size_t)p->num_chunks * L.bpc, 256);
    off += L.bmap_bytes;
    L.marks_off = off;
    L.marks_bytes = align_up((size_t)p->num_chunks * L.bpc, 256);
    off += L.marks_bytes;
    L.zero_off = off;
    L.head_off = off;
    off += 256;
    L.tiles_off = off;
    L.tiles_bytes = align_up((size_t)p->num_chunks * sizeof(int32_t), 256);
    off += L.tiles_bytes;
    L.arrive_off = off;
    L.arrive_bytes = align_up((size_t)p->num_chunks * ((L.nbz + 7) / 8) * ((L.nby + 7) / 8) * L.wpr * sizeof(int32_t), 256);
    off += L.arrive_bytes;
    L.loss_off = off;
    L.loss_bytes = align_up((size_t)kLossSlots * 8 * sizeof(double), 256);
    off += L.loss_bytes;
    L.zero_bytes = off - L.zero_off;
    L.list_off = off;
    L.list_bytes = align_up((size_t)(p->num_locs > 0 ? p->num_locs : 0) * F * 2 * sizeof(int32_t), 256);
    off += L.list_bytes;
    L.hits_off = off;
    L.hits_bytes = align_up((size_t)p->num_chunks * F * p->width * p->height * sizeof(int32_t), 256);
    off += L.hits_bytes;
    L.det_off = off;
    L.det_bytes = 0;
    if (p->flags & SPSG_FLAG_DETERMINISTIC)
        L.det_bytes = det_loss_partials_bytes((long long)p->num_chunks * F * p->width * p->height);
    off += L.det_bytes;
    const bool all = (p->flags & SPSG_FLAG_ALL_PIXELS) != 0;
    const size_t rows = (size_t)(p->num_locs > 0 ? p->num_locs : 0) * F;
    const size_t pixels = (size_t)p->num_chunks * F * p->width * p->height;
    L.seg_head_off = off;
    L.seg_head_bytes = all ? 256 : 0;
    off += L.seg_head_bytes;
    L.seg_end_off = off;
    L.seg_end_bytes = all ? align_up(rows * sizeof(int32_t), 256) : 0;
    off += L.seg_end_bytes;
    L.seg_pix_off = off;
    L.seg_pix_bytes = all ? align_up(pixels * sizeof(int32_t), 256) : 0;
    off += L.seg_pix_bytes;
    L.seg_long_off = off;
    L.seg_long_bytes = all && (p->flags & SPSG_FLAG_DETERMINISTIC) ? align_up((pixels / (kSegWarpSort + 1) + 1) * sizeof(int32_t), 256) : 0;
    off += L.seg_long_bytes;
    L.total = off;
    return L;
}
