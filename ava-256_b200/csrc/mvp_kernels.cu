// mvp_kernels.cu -- B200 (sm_100a) volumetric-primitive raymarcher: accel build, forward, backward.
//
// Replaces (semantics, not code) /root/reference/extensions/mvpraymarch/{mvpraymarch_kernel.cu, bvh.cu,
// mvpraymarch_subset_kernel.h, utils.h, primtransf.h, primsampler.h, primaccum.h}.  See DESIGN.md for the
// data layout and the per-kernel rooflines.  Design in one paragraph:
//
//   * No BVH.  The reference finds each warp's candidate slabs by a DFS over a 2K-1 node AABB heap
//     (utils.h:719-815), per warp, per kernel.  Here a view's camera is recovered from its ray field
//     (fit_camera_kernel, verified against every ray), every slab OBB is projected to a pixel rectangle
//     (prim_setup_kernel) and rectangles are bucketed into 4-pixel-high tile rows in DFS-rank order
//     (row_lists_kernel).  A warp (= one 8x4 pixel tile, the reference's warp footprint) scans its row's
//     bucket, keeps rectangles that overlap its 8 columns, and runs the reference's *exact* per-lane slab
//     test on them -- so list membership, per-ray [t_enter,t_exit] and the 512 cap are the reference's.
//     Views whose rays are not a pinhole grid fall back to "every slab is a candidate" (correct, slow).
//   * Interval marching.  The reference re-transforms every listed slab at every step.  Here each list entry
//     carries the warp's step interval; per step one ballot per 32 list slots finds the active slabs and only those
//     are transformed; stretches without an active slab are skipped.  Ray position and t advance incrementally in
//     fp32 exactly as in the reference (mvpraymarch_subset_kernel.h:95-96) so validity decisions match bit for bit.
//   * Sample compaction.  Valid samples are queued in shared memory and the gather/interpolation (forward) or the
//     whole adjoint (backward) runs on full batches of 32 samples; forward composites per ray in queue order.
//   * Backward is slab-major: forward records, per ray, the saturating sample (step, rank) and the alpha before it,
//     which removes the only order dependence (primaccum.h:81-98).  Each warp walks one slab at a time (every lane its
//     own step interval), keeps factored transform gradients in registers, reduces them with a 16-value butterfly and
//     issues one atomic per value per (warp, slab); payload gradients go out as 128-bit vector reductions
//     (red.global.add.v4.f32) instead of 32 scalar atomics per sample.
//   * The tile row's bucket (second level: the row's entries that touch a group of 8 tile columns) is staged through shared
//     memory by the TMA engine (cp.async.bulk + mbarrier); list entries carry step intervals derived from a bound on the
//     fp drift of the marched positions.
//   * In gradient mode the forward saves each tile's list and each ray's first step in the workspace; the backward loads
//     them instead of repeating the bucket scan and the exact slab tests.
//   * Two kernels per pass: the fast one (256-entry shared-memory lists) renders every tile whose list fits -- all of them in
//     the benchmark scene -- and appends the others to an overflow list; a small persistent 512-entry kernel (the reference's
//     cap, utils.h:779-781) then renders those.
//   * Backward register diet: the slab record and, optionally, the per-lane state that is only touched between batches live in
//     shared memory, so the batch adjoint (the kernel's register peak) sees few live values.
//
// Arithmetic mirrors the reference's fp32 operation order where a step function of the result exists
// (transform + strict validity, slab test, lattice snap, saturation); -use_fast_math is on like the reference.

#ifdef MVP_CPU_EMUL
// Test-only host build (tests/emul/): the kernels below compiled with g++ on top of a CPU emulation of warps, blocks and
// shared memory, so the CPU test suite can run this file's logic against the oracle.  Not part of the product library.
#include "cuda_emul.h"
#else
#include <cuda_runtime.h>
#include <math_constants.h>
#endif
#include <stdint.h>
#include <stdlib.h>

#include "mvpraymarch_b200.h"
#include "raygen.h"
#include <stddef.h>

// C-ABI layout pins (the ctypes mirror in ava-256_b200/lib.py and INTEGRATION.md are checked against the same numbers)
static_assert(sizeof(mvp_shape) == 28, "mvp_shape layout");
static_assert(sizeof(mvp_camera) == 40, "mvp_camera layout");
static_assert(sizeof(mvp_forward_args) == 272 && offsetof(mvp_forward_args, camera) == 232 && offsetof(mvp_forward_args, raypos) == 48 && offsetof(mvp_forward_args, workspace_bytes) == 136 &&
                  offsetof(mvp_forward_args, algo) == 164, "mvp_forward_args layout");
static_assert(sizeof(mvp_backward_args) == 272 && offsetof(mvp_backward_args, camera) == 232 && offsetof(mvp_backward_args, grad_rayrgba) == 104 && offsetof(mvp_backward_args, workspace_bytes) == 168 &&
                  offsetof(mvp_backward_args, algo) == 204, "mvp_backward_args layout");

// experiment knobs (defaults = measured best)
#ifndef MVP_BWD_LO_SLACK
#define MVP_BWD_LO_SLACK 0.f   // one step of slack on each side: the strictly-inside range (1.f / 0.f) is 2 % faster but drops
#define MVP_BWD_HI_SLACK 1.f   // ~1e-3 of the samples (on slab faces, |dfade/dy| still 2 % of an interior sample): grads off by 1e-4
#endif
#ifndef MVP_CHUNK
#define MVP_CHUNK 16
#endif

namespace {

constexpr int kMaxHit = 512;      // utils.h:779-781 (template argument hard-wired at mvpraymarch_kernel.cu:33)
constexpr int kTileW = 8;         // warp footprint of the reference's default block (8,16): 8 x 4 pixels
constexpr int kTileH = 4;
#ifndef MVP_BLK_TX
#define MVP_BLK_TX 2
#endif
#ifndef MVP_XBUCKETS
#define MVP_XBUCKETS 1   // 1: second bucketing level in x (groups of 8 tile columns): a tile scans ~45 instead of ~350 bucket
                          // entries (-80 % of the chunk scans).  Measured on B200 (round 2): forward 2.68 vs 2.80 ms per 8 views
#endif
#ifndef MVP_LIST_MARGIN
#define MVP_LIST_MARGIN 1   // 1: step intervals of the tile lists from a bound on the fp drift of the marched positions instead of a
                            // whole step of slack on each side: -26 % forward events.  Measured on B200 (round 2, with the zero-scale fix, all
                            // GPU tests green): forward 2.70 vs 2.80, backward 3.47 vs 3.69 ms per 8 views; both knobs: 2.59 / 3.46
#endif
#ifndef MVP_LIST_CAP_MIN
#define MVP_LIST_CAP_MIN 4096
#endif
#ifndef MVP_LIST_CAP_PER_TILE
#define MVP_LIST_CAP_PER_TILE 24   // average saved entries per tile the workspace provides (C3 scene: 8 on average)
#endif
#ifndef MVP_LIST_REUSE
#define MVP_LIST_REUSE 1   // the forward (gradient mode) saves each tile's slab list and each ray's first step, the backward loads
                           // them instead of rebuilding.  Measured on B200: backward 3.44 vs 4.23 ms per 8 views (-19 %)
#endif
#ifndef MVP_WARPS
#define MVP_WARPS 4
#endif
constexpr int kWarps = MVP_WARPS;   // warps (tiles) per CTA: 2 measured 4-5 % slower (fwd and bwd); 8 overflows the 48 KB static smem of the CAP=512 variants
constexpr int kBlkTX = MVP_BLK_TX;   // ... arranged kBlkTX x kBlkTY tiles (2 x 2 = 16 x 8 pixels: measured best)
constexpr int kBlkTY = kWarps / kBlkTX;
constexpr int kMaskSteps = MVP_CHUNK;   // backward: sweep steps per chunk of slab start order
constexpr int kRowCapMax = 2048;  // entries per tile-row bucket before the row falls back to scanning all slabs
constexpr int kRing = 64;        // sample queue / ring per warp (forward and backward; power of two, >= 2 * 32)
#ifndef MVP_PREFETCH
#define MVP_PREFETCH 0   // measured: +1 % forward speed but +50 % DRAM reads (slabs of rays that saturate earlier are fetched in vain)
#endif
#ifndef MVP_FASTCAP
#define MVP_FASTCAP 256
#endif
#ifndef MVP_BWD_SMEMREC
#define MVP_BWD_SMEMREC 1   // backward: the current slab's 64-byte record lives in shared memory; the step loop re-reads it after every
                            // batch adjoint and the adjoint reads what it needs from there, so the record's 15 registers are not
                            // live across the adjoint (the kernel's register peak)
#endif
#ifndef MVP_TILE_CLOCKS
#define MVP_TILE_CLOCKS 0   // diagnostics build only: the forward kernel records (start, duration) in SM clock cycles and the SM id per tile
#endif
#ifndef MVP_CTA_ORDER_MIN
#define MVP_CTA_ORDER_MIN 0    // > 0: only CTAs of cost class >= this are moved to the front, the others keep the grid order among
                               // themselves.  Measured (30 / 40 / 50): no better than the full sort for either kernel
#endif
#ifndef MVP_CTA_ORDER_MAXVIEWS
#define MVP_CTA_ORDER_MAXVIEWS 16   // the cost order (and the estimate behind it) is used only for launches of at most this many views.
                                    // Measured on B200, sorted vs grid order: forward -10..-14 % and backward -2.6 % at 10 views per launch
                                    // (one rank of an 8-GPU run); at 40 and 80 views the differences (-3 % .. +2 %) are within the
                                    // box-to-box noise: long launches have no tail to speak of
#endif
#ifndef MVP_CTA_ORDER
#define MVP_CTA_ORDER 1   // 1: the render kernels' CTAs run in descending order of a cost estimate (candidate slabs of the CTA's tile rows),
                          // over all views of the launch: the expensive silhouette tiles -- a single warp can be busy for ~1 ms with
                          // one of them -- start first and the cheap background tiles fill in behind, instead of a launch ending with
                          // a few long-running warps.  Matters for small launches (10 views per rank at 8 GPUs); 0: plain grid order
#endif
#ifndef MVP_BWD_LANESMEM
#define MVP_BWD_LANESMEM 0   // backward: per-lane state that is only touched between batches (ray origin / t-range, sweep limits, chunk
                             // base position, the 12 transform-gradient accumulators) lives in shared memory instead of registers
#endif
#if MVP_XBUCKETS
constexpr int kGrpTiles = 8;       // tile columns per x-group
constexpr int kGrpCap = 1024;     // group-bucket entries per tile row; groups that do not fit keep using the row bucket
#endif
#ifndef MVP_FWD_FASTCAP
#define MVP_FWD_FASTCAP MVP_FASTCAP
#endif
#ifndef MVP_BWD_FASTCAP
#define MVP_BWD_FASTCAP MVP_FASTCAP
#endif
constexpr int kFastCapF = MVP_FWD_FASTCAP;   // shared-memory list capacity of the common-case render kernels (forward / backward); a tile whose
constexpr int kFastCapB = MVP_BWD_FASTCAP;   // list is longer goes to the 512-entry kernel of that pass (the backward's may be the smaller one)
#ifndef MVP_SMEM_UNION
#define MVP_SMEM_UNION 1   // 1: the bucket staging buffer (used only while a tile's list is built) shares its shared memory with the sample
                           // queue (used only afterwards): 512 bytes less per warp.  Measured on B200 (round 2): forward 2.096 vs 2.120 ms per
                           // 8 views, 10.475 vs 10.610 per 40; backward unchanged
#endif
#ifndef MVP_FWD_RING
#define MVP_FWD_RING 1   // 1: the forward's sample queue is a ring of two 32-entry halves -- a flush always takes exactly one half, so the
                          // head alternates between 0 and 32 and nothing is ever moved; 0: the queue is compacted to the front after every
                          // flush (two shared-memory passes and three warp barriers per batch)
#endif
#ifndef MVP_FWD_CARVEOUT
#define MVP_FWD_CARVEOUT 0   // > 0: preferred shared-memory carve-out (percent of the maximum, cudaFuncAttributePreferredSharedMemoryCarveout) of the
#endif                       // fast render kernels; 0 leaves the driver's choice.  The kernels live off L1 hits: what is not carved out is L1
#ifndef MVP_BWD_CARVEOUT
#define MVP_BWD_CARVEOUT 43   // 100 KB of shared memory (4 CTAs need 81): the driver's own choice is 132 KB.  Measured: backward 2.821 vs 2.835 ms
#endif                        // per 8 views, 14.187 vs 14.257 per 40.  The carve-out matters little either way (forward at 100 KB instead of
                              // 132: +-0; at 164 KB: +2 %; backward at 64 KB: +-0): the kernels are issue bound, not L1-capacity bound
constexpr int kBig = 1 << 30;
constexpr int kCostClasses = 64;   // cost classes of the CTA ordering (counting sort)
#ifndef MVP_BWD_MINB
#define MVP_BWD_MINB 4   // resident CTAs per SM the backward kernel is compiled for (register cap 65536 / (128 * MINB))
#endif
#ifndef MVP_FWD_MINB
#define MVP_FWD_MINB 7   // 72 registers: one CTA less per SM than at 64, but no re-materialised address math per event (measured -2 %)
#endif

struct Cam {          // 64 B per view
    float o[3];
    int ok;           // fit succeeded (consumers also check bad[n] == 0)
    float minv[9];    // pixel (w,h,1) ~ minv * (P - o)
    float pad[3];
};

struct __align__(8) RowEntry { int k; unsigned xr; };   // xr = x0 | x1 << 16  (pixels, inclusive)

struct Layout {
    size_t cam, raycam, bad, pack, rx, ry, rowcnt, rowlist, heavycnt, heavylist, ctaorder, ctahist, tilecnt, blky, rankof, tileclk, total;
    int R, rowcap;
#if MVP_XBUCKETS
    size_t grphdr, grplist;
    int NG;           // x-groups per tile row
#endif
#if MVP_LIST_REUSE
    size_t tilehdr, listbuf, listcur, rayj0;
    int listcap;      // saved list entries per view (tiles that do not fit are rebuilt by the backward)
#endif
};

__host__ __device__ inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

__host__ inline Layout make_layout(const mvp_shape &s) {
    Layout L;
    L.R = (s.H + kTileH - 1) / kTileH;
    L.rowcap = ((s.K < kRowCapMax ? s.K : kRowCapMax) + 1) & ~1;   // even: 16-byte aligned buckets (TMA bulk copies)
    size_t off = 0;
    L.cam = off;     off = align256(off + (size_t)s.N * sizeof(Cam));
    L.raycam = off;  off = align256(off + (size_t)s.N * 4 * sizeof(float4));
    L.bad = off;     off = align256(off + (size_t)s.N * sizeof(int));
    L.pack = off;    off = align256(off + (size_t)s.N * s.K * 64);
    L.rx = off;      off = align256(off + (size_t)s.N * s.K * 4);
    L.ry = off;      off = align256(off + (size_t)s.N * s.K * 4);
    L.blky = off;    off = align256(off + (size_t)s.N * ((s.K + 31) / 32) * 4);
    L.rankof = off;  off = align256(off + (size_t)s.N * s.K * 4);
    L.rowcnt = off;  off = align256(off + (size_t)s.N * L.R * 4);
    L.rowlist = off; off = align256(off + (size_t)s.N * L.R * L.rowcap * sizeof(RowEntry));
    {
        const size_t ctas = (size_t)s.N * (((s.H + kTileH - 1) / kTileH + kBlkTY - 1) / kBlkTY) * (((s.W + kTileW - 1) / kTileW + kBlkTX - 1) / kBlkTX);
        L.ctaorder = off; off = align256(off + ctas * sizeof(int));
        L.ctahist = off;  off = align256(off + 2 * kCostClasses * sizeof(int));
        L.tilecnt = off;  off = align256(off + (size_t)s.N * ((s.H + kTileH - 1) / kTileH) * ((s.W + kTileW - 1) / kTileW) * sizeof(unsigned short));
    }
#if MVP_TILE_CLOCKS
    L.tileclk = off; off = align256(off + (size_t)s.N * ((s.H + kTileH - 1) / kTileH) * ((s.W + kTileW - 1) / kTileW) * 4 * sizeof(long long));
#else
    L.tileclk = 0;
#endif
    L.heavycnt = off; off = align256(off + sizeof(int));
    L.heavylist = off; off = align256(off + (size_t)s.N * ((s.H + kTileH - 1) / kTileH) * ((s.W + kTileW - 1) / kTileW) * sizeof(int));
#if MVP_XBUCKETS
    L.NG = ((s.W + kTileW - 1) / kTileW + kGrpTiles - 1) / kGrpTiles;
    L.grphdr = off;  off = align256(off + (size_t)s.N * L.R * L.NG * sizeof(int2));
    L.grplist = off; off = align256(off + (size_t)s.N * L.R * kGrpCap * sizeof(RowEntry));
#endif
#if MVP_LIST_REUSE
    {
        const size_t tiles = (size_t)((s.H + kTileH - 1) / kTileH) * ((s.W + kTileW - 1) / kTileW);
        const size_t cap = tiles * MVP_LIST_CAP_PER_TILE < MVP_LIST_CAP_MIN ? MVP_LIST_CAP_MIN : tiles * MVP_LIST_CAP_PER_TILE;
        L.listcap = (int)(cap < (size_t)0x3fffffff ? cap : (size_t)0x3fffffff);
        L.tilehdr = off; off = align256(off + (size_t)s.N * tiles * sizeof(int2));
        L.listbuf = off; off = align256(off + (size_t)s.N * L.listcap * sizeof(int2));
        L.listcur = off; off = align256(off + (size_t)s.N * sizeof(int));
        L.rayj0 = off;   off = align256(off + (size_t)s.N * s.H * s.W * sizeof(int));
    }
#endif
    L.total = off;
    return L;
}

// DFS leaf order of the reference's implicit heap (utils.h:740-742, 788): leaves are visited in the order
// k = kstart, kstart+1, ..., K-1, 0, ..., kstart-1 with kstart = nextpow2(K) - K  (0 when K is a power of two).
__host__ __device__ inline int dfs_kstart(int K) {
    int P = 1;
    while (P < K) P <<= 1;
    return P - K;
}

// Marching order of a view's slabs.  Default ("fixedorder"): the rotation above.  With an explicit order (usebvh=True: ascending
// Morton code of the centres, the `sortedobjid` of mvpraymarch.py:46-55) leaf i of the heap holds slab order[i] (rankof = its
// inverse) -- an indirection in the accel build and two lookups in the render kernels instead of gathering the primitive
// tensors (134 MB of payload per view) into that order.
__device__ __forceinline__ int slab_at_rank(const int *__restrict__ order, int K, int kstart, int j) {
    int leaf = j + kstart;                       // DFS visits the leaves of the implicit heap in this rotated sequence ...
    if (leaf >= K) leaf -= K;
    return order ? order[leaf] : leaf;           // ... and leaf i holds slab sortedobjid[i]
}
__device__ __forceinline__ int rank_of_slab(const int *__restrict__ rankof, int K, int kstart, int k) {
    int r = (rankof ? rankof[k] : k) - kstart;
    if (r < 0) r += K;
    return r;
}

// rankof[n][order[n][j]] = j
__global__ void __launch_bounds__(256) invert_order_kernel(size_t NK, int K, const int *__restrict__ order, int *__restrict__ rankof) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= NK) return;
    const size_t n = i / (size_t)K;
    rankof[n * K + order[i]] = (int)(i - n * K);
}

// ------------------------------------------------------------------------------------------------------
// 1. camera fit: D(w,h) = A + B w + C h  with raydir(w,h) = normalize(D); verified on every ray.
// ------------------------------------------------------------------------------------------------------
constexpr int kFitThreads = 256;
constexpr int kFitRaysPerThread = 8;

__global__ void __launch_bounds__(kFitThreads) fit_camera_kernel(int H, int W, const float *__restrict__ raypos,
                                                                 const float *__restrict__ raydir, Cam *cam, int *bad) {
    const int n = blockIdx.y;
    const size_t HW = (size_t)H * W;
    const float *rp = raypos + (size_t)n * HW * 3;
    const float *rd = raydir + (size_t)n * HW * 3;
    __shared__ float s_minv[9];
    __shared__ float s_o[3];
    __shared__ int s_ok;
    if (threadIdx.x == 0) {
        int ok = (W >= 2 && H >= 2);
        double mi[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        if (ok) {
            double d00[3], d10[3], d01[3], d11[3];
            const size_t i00 = 0, i10 = (size_t)(W - 1), i01 = (size_t)(H - 1) * W, i11 = HW - 1;
            for (int i = 0; i < 3; ++i) {
                d00[i] = rd[i00 * 3 + i]; d10[i] = rd[i10 * 3 + i]; d01[i] = rd[i01 * 3 + i]; d11[i] = rd[i11 * 3 + i];
            }
            // [d10 d01 -d00] (b,c,a)^T = d11
            double m[9] = {d10[0], d01[0], -d00[0], d10[1], d01[1], -d00[1], d10[2], d01[2], -d00[2]};
            double det = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
            if (!(fabs(det) > 1e-12)) ok = 0;
            double b = 0, c = 0, a = 0;
            if (ok) {
                double id = 1.0 / det;
                b = id * (d11[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (d11[1] * m[8] - m[5] * d11[2]) + m[2] * (d11[1] * m[7] - m[4] * d11[2]));
                c = id * (m[0] * (d11[1] * m[8] - m[5] * d11[2]) - d11[0] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * d11[2] - d11[1] * m[6]));
                a = id * (m[0] * (m[4] * d11[2] - d11[1] * m[7]) - m[1] * (m[3] * d11[2] - d11[1] * m[6]) + d11[0] * (m[3] * m[7] - m[4] * m[6]));
                if (!(a > 1e-9 && b > 1e-9 && c > 1e-9) || !isfinite(a + b + c)) ok = 0;
            }
            if (ok) {
                double A[3], B[3], C[3];
                for (int i = 0; i < 3; ++i) {
                    A[i] = a * d00[i];
                    B[i] = (b * d10[i] - A[i]) / (double)(W - 1);
                    C[i] = (c * d01[i] - A[i]) / (double)(H - 1);
                }
                // M = [B C A] (columns); invert
                double M[9] = {B[0], C[0], A[0], B[1], C[1], A[1], B[2], C[2], A[2]};
                double dm = M[0] * (M[4] * M[8] - M[5] * M[7]) - M[1] * (M[3] * M[8] - M[5] * M[6]) + M[2] * (M[3] * M[7] - M[4] * M[6]);
                if (!(fabs(dm) > 1e-30) || !isfinite(dm)) ok = 0;
                else {
                    double im = 1.0 / dm;
                    mi[0] = (M[4] * M[8] - M[5] * M[7]) * im; mi[1] = (M[2] * M[7] - M[1] * M[8]) * im; mi[2] = (M[1] * M[5] - M[2] * M[4]) * im;
                    mi[3] = (M[5] * M[6] - M[3] * M[8]) * im; mi[4] = (M[0] * M[8] - M[2] * M[6]) * im; mi[5] = (M[2] * M[3] - M[0] * M[5]) * im;
                    mi[6] = (M[3] * M[7] - M[4] * M[6]) * im; mi[7] = (M[1] * M[6] - M[0] * M[7]) * im; mi[8] = (M[0] * M[4] - M[1] * M[3]) * im;
                    for (int i = 0; i < 9; ++i) if (!isfinite(mi[i])) ok = 0;
                }
            }
        }
        for (int i = 0; i < 9; ++i) s_minv[i] = (float)mi[i];
        for (int i = 0; i < 3; ++i) s_o[i] = rp[i];
        s_ok = ok;
    }
    __syncthreads();
    int fail = 0;
    if (s_ok) {
        const float m0 = s_minv[0], m1 = s_minv[1], m2 = s_minv[2], m3 = s_minv[3], m4 = s_minv[4], m5 = s_minv[5],
                    m6 = s_minv[6], m7 = s_minv[7], m8 = s_minv[8];
        const float ox = s_o[0], oy = s_o[1], oz = s_o[2];
        size_t base = (size_t)blockIdx.x * (kFitThreads * kFitRaysPerThread);
#pragma unroll
        for (int it = 0; it < kFitRaysPerThread; ++it) {
            size_t r = base + (size_t)it * kFitThreads + threadIdx.x;
            if (r < HW) {
                float px_ = __ldg(rp + r * 3 + 0), py_ = __ldg(rp + r * 3 + 1), pz_ = __ldg(rp + r * 3 + 2);
                float dx = __ldg(rd + r * 3 + 0), dy = __ldg(rd + r * 3 + 1), dz = __ldg(rd + r * 3 + 2);
                int w = (int)(r % (size_t)W), h = (int)(r / (size_t)W);
                float qx = m0 * dx + m1 * dy + m2 * dz, qy = m3 * dx + m4 * dy + m5 * dz, qz = m6 * dx + m7 * dy + m8 * dz;
                float u = __fdiv_rn(qx, qz), v = __fdiv_rn(qy, qz);
                bool good = (px_ == ox) && (py_ == oy) && (pz_ == oz) && (qz > 0.f) && (fabsf(u - (float)w) < 0.05f) &&
                            (fabsf(v - (float)h) < 0.05f);
                fail |= !good;
            }
        }
    } else {
        fail = 1;
    }
    fail = __syncthreads_or(fail);
    if (threadIdx.x == 0) {
        if (fail) atomicOr(bad + n, 1);
        if (blockIdx.x == 0) {
            Cam c;
            for (int i = 0; i < 3; ++i) c.o[i] = s_o[i];
            c.ok = s_ok;
            for (int i = 0; i < 9; ++i) c.minv[i] = s_minv[i];
            c.pad[0] = c.pad[1] = c.pad[2] = 0.f;
            cam[n] = c;
        }
    }
}

// 1b. The same record from the camera parameters themselves (mvp_camera): D(w,h) = row2 + row0 (w - cx) / fx + row1 (h - cy) / fy is a
//     pinhole grid by construction, so there is nothing to fit and nothing to verify -- no pass over a ray field that, in this mode,
//     does not exist.  Also writes the record the render kernels generate their rays from (raygen.h).  One thread per view.
__global__ void __launch_bounds__(128) cam_params_kernel(int N, const float *__restrict__ viewpos, const float *__restrict__ viewrot,
                                                         const float *__restrict__ focal, const float *__restrict__ princpt, float volradius,
                                                         Cam *cam, int *bad, float4 *raycam) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float *R = viewrot + (size_t)n * 9;
    const float fx = focal[n * 2 + 0], fy = focal[n * 2 + 1], cx = princpt[n * 2 + 0], cy = princpt[n * 2 + 1];
    Cam c;
    // ray origin exactly as the generator computes it (utils_kernel.cu:32)
    c.o[0] = __fdiv_rn(viewpos[n * 3 + 0], volradius); c.o[1] = __fdiv_rn(viewpos[n * 3 + 1], volradius); c.o[2] = __fdiv_rn(viewpos[n * 3 + 2], volradius);
    raycam[(size_t)n * 4 + 0] = make_float4(c.o[0], c.o[1], c.o[2], R[0]);
    raycam[(size_t)n * 4 + 1] = make_float4(R[1], R[2], R[3], R[4]);
    raycam[(size_t)n * 4 + 2] = make_float4(R[5], R[6], R[7], R[8]);
    raycam[(size_t)n * 4 + 3] = make_float4(cx, cy, fx, fy);
    int ok = 1;
    double mi[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    double A[3], B[3], C[3];
    for (int i = 0; i < 3; ++i) {
        B[i] = (double)R[i] / (double)fx;
        C[i] = (double)R[3 + i] / (double)fy;
        A[i] = (double)R[6 + i] - B[i] * (double)cx - C[i] * (double)cy;
    }
    // M = [B C A] (columns); pixel (w, h, 1) ~ M^-1 (P - o)
    const double M[9] = {B[0], C[0], A[0], B[1], C[1], A[1], B[2], C[2], A[2]};
    const double dm = M[0] * (M[4] * M[8] - M[5] * M[7]) - M[1] * (M[3] * M[8] - M[5] * M[6]) + M[2] * (M[3] * M[7] - M[4] * M[6]);
    if (!(fabs(dm) > 1e-30) || !isfinite(dm)) ok = 0;
    else {
        const double im = 1.0 / dm;
        mi[0] = (M[4] * M[8] - M[5] * M[7]) * im; mi[1] = (M[2] * M[7] - M[1] * M[8]) * im; mi[2] = (M[1] * M[5] - M[2] * M[4]) * im;
        mi[3] = (M[5] * M[6] - M[3] * M[8]) * im; mi[4] = (M[0] * M[8] - M[2] * M[6]) * im; mi[5] = (M[2] * M[3] - M[0] * M[5]) * im;
        mi[6] = (M[3] * M[7] - M[4] * M[6]) * im; mi[7] = (M[1] * M[6] - M[0] * M[7]) * im; mi[8] = (M[0] * M[4] - M[1] * M[3]) * im;
        for (int i = 0; i < 9; ++i) if (!isfinite(mi[i])) ok = 0;
    }
    if (!isfinite(c.o[0]) || !isfinite(c.o[1]) || !isfinite(c.o[2])) ok = 0;
    c.ok = ok;
    for (int i = 0; i < 9; ++i) c.minv[i] = (float)mi[i];
    c.pad[0] = c.pad[1] = c.pad[2] = 0.f;
    cam[n] = c;
    bad[n] = ok ? 0 : 1;          // a degenerate camera (focal 0, non-finite) falls back to "every slab is a candidate", like a failed fit
}

// ------------------------------------------------------------------------------------------------------
// 2. per-slab record + pixel rectangle
//    record (4 x float4): (pos.xyz, s.x) (R row0, s.y) (R row1, s.z) (R row2, 0)
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) prim_setup_kernel(int N, int K, int H, int W, int pview, const float *__restrict__ primpos,
                                                         const float *__restrict__ primrot, const float *__restrict__ primscale,
                                                         const Cam *__restrict__ cam, const int *__restrict__ bad,
                                                         float4 *__restrict__ pack, unsigned *__restrict__ rx, unsigned *__restrict__ ry) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * K) return;
    const int n = (int)(i / (size_t)K);
    const size_t ip = pview ? i : i - (size_t)n * K;     // index of the slab in the primitive tensors / record array
    const float *pp = primpos + ip * 3, *pr = primrot + ip * 9, *ps = primscale + ip * 3;
    float p0 = pp[0], p1 = pp[1], p2 = pp[2];
    float r[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) r[j] = pr[j];
    float s0 = ps[0], s1 = ps[1], s2 = ps[2];
    if (pview || n == 0) {
        pack[ip * 4 + 0] = make_float4(p0, p1, p2, s0);
        pack[ip * 4 + 1] = make_float4(r[0], r[1], r[2], s1);
        pack[ip * 4 + 2] = make_float4(r[3], r[4], r[5], s2);
        pack[ip * 4 + 3] = make_float4(r[6], r[7], r[8], 0.f);
    }

    // rectangle: full screen unless the view is a verified pinhole and all 8 corners are on one side of it
    int x0 = 0, x1 = W - 1, y0 = 0, y1 = H - 1;
    const Cam c = cam[n];
    if (c.ok && bad[n] == 0) {
        float e0 = __fdiv_rn(1.f, s0), e1 = __fdiv_rn(1.f, s1), e2 = __fdiv_rn(1.f, s2);
        float umin = CUDART_INF_F, umax = -CUDART_INF_F, vmin = CUDART_INF_F, vmax = -CUDART_INF_F;
        float zmin = CUDART_INF_F, zmax = -CUDART_INF_F;
        bool nan = false;
#pragma unroll
        for (int cidx = 0; cidx < 8; ++cidx) {
            float a = (cidx & 1) ? e0 : -e0, b = (cidx & 2) ? e1 : -e1, d = (cidx & 4) ? e2 : -e2;
            // world corner = R (c / s) + pos   (primtransf.h:12-63)
            float wx = r[0] * a + r[1] * b + r[2] * d + p0 - c.o[0];
            float wy = r[3] * a + r[4] * b + r[5] * d + p1 - c.o[1];
            float wz = r[6] * a + r[7] * b + r[8] * d + p2 - c.o[2];
            float qx = c.minv[0] * wx + c.minv[1] * wy + c.minv[2] * wz;
            float qy = c.minv[3] * wx + c.minv[4] * wy + c.minv[5] * wz;
            float qz = c.minv[6] * wx + c.minv[7] * wy + c.minv[8] * wz;
            float u = __fdiv_rn(qx, qz), v = __fdiv_rn(qy, qz);
            nan |= !(u == u) || !(v == v) || !(qz == qz);
            umin = fminf(umin, u); umax = fmaxf(umax, u); vmin = fminf(vmin, v); vmax = fmaxf(vmax, v);
            zmin = fminf(zmin, qz); zmax = fmaxf(zmax, qz);
        }
        // lines, not half-lines (utils.h:747-755 has no t >= 0 clip): a slab entirely behind the pinhole projects
        // through it just the same; only a slab straddling the plane qz = 0 has an unbounded footprint.
        const float zeps = 1e-6f * fmaxf(fabsf(zmin), fabsf(zmax));
        if (!nan && (zmin > zeps || zmax < -zeps)) {
            float fx0 = fmaxf(floorf(umin) - 1.f, 0.f), fx1 = fminf(ceilf(umax) + 1.f, (float)(W - 1));
            float fy0 = fmaxf(floorf(vmin) - 1.f, 0.f), fy1 = fminf(ceilf(vmax) + 1.f, (float)(H - 1));
            if (fx0 > fx1 || fy0 > fy1) { x0 = 1; x1 = 0; y0 = 1; y1 = 0; }   // off screen: empty
            else { x0 = (int)fx0; x1 = (int)fx1; y0 = (int)fy0; y1 = (int)fy1; }
        }
    }
    rx[i] = (unsigned)x0 | ((unsigned)x1 << 16);
    ry[i] = (unsigned)y0 | ((unsigned)y1 << 16);
}

// ------------------------------------------------------------------------------------------------------
// 3. tile-row buckets in DFS-rank order (deterministic ordered compaction; one CTA per (row, view))
// ------------------------------------------------------------------------------------------------------
// y range (pixels) of every block of 32 slabs consecutive in DFS rank: the bucket kernels test a block before its slabs, so a
// tile row only touches the ~10-20 % of the blocks that can reach it (slabs follow the UV grid: consecutive ranks are neighbours).
__global__ void __launch_bounds__(256) block_ranges_kernel(int K, const unsigned *__restrict__ ry, const int *__restrict__ order,
                                                           int ostride, unsigned *__restrict__ blky) {
    const int lane = threadIdx.x & 31;
    const int NB = (K + 31) / 32;
    const int blk = blockIdx.x * 8 + (threadIdx.x >> 5), n = blockIdx.y;
    if (blk >= NB) return;
    const int kstart = dfs_kstart(K);
    const int j = blk * 32 + lane;
    int y0 = 0xffff, y1 = -1;
    if (j < K) {
        const int k = slab_at_rank(order ? order + (size_t)n * ostride : nullptr, K, kstart, j);
        const unsigned yr = __ldg(ry + (size_t)n * K + k);
        const int a = (int)(yr & 0xffffu), b = (int)(yr >> 16);
        if (a <= b) { y0 = a; y1 = b; }
    }
    y0 = __reduce_min_sync(0xffffffffu, y0);
    y1 = __reduce_max_sync(0xffffffffu, y1);
    if (lane == 0) blky[(size_t)n * NB + blk] = (y1 < 0) ? 1u : ((unsigned)y0 | ((unsigned)y1 << 16));   // 1 | 0 << 16: empty
}

constexpr int kRowThreads = 256;          // 8 warps = 8 tile rows per CTA

// One WARP per (tile row, view): it walks the view's slabs in DFS-rank order, 32 at a time, and appends those whose rectangle
// touches the row -- an ordered compaction that needs nothing but a ballot per step (no block-wide barrier: the round-1 kernel
// spent its time in three __syncthreads per 256 slabs).  The 8 warps of a CTA read the same rectangle arrays (L1 hits).
__global__ void __launch_bounds__(kRowThreads) row_lists_kernel(int K, int R, int rowcap, int TXn,
                                                                const unsigned *__restrict__ rx, const unsigned *__restrict__ ry,
                                                                const unsigned *__restrict__ blky, const int *__restrict__ order, int ostride,
                                                                int *__restrict__ rowcnt, RowEntry *__restrict__ rowlist
#if MVP_XBUCKETS
                                                                , int NG, int2 *__restrict__ grphdr, RowEntry *__restrict__ grplist,
                                                                unsigned short *__restrict__ tilecnt   // NULL: no cost estimate wanted
#endif
                                                                ) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = blockIdx.x * (kRowThreads / 32) + warp, n = blockIdx.y;
    if (row >= R) return;                      // warps are independent
    const int ylo = row * kTileH, yhi = ylo + kTileH - 1;
    const unsigned *rxn = rx + (size_t)n * K, *ryn = ry + (size_t)n * K;
    RowEntry *out = rowlist + ((size_t)n * R + row) * rowcap;
    const int kstart = dfs_kstart(K);
    const int *ordn = order ? order + (size_t)n * ostride : nullptr;
    const unsigned below = (1u << lane) - 1u;
    int total = 0;
    const int NB = (K + 31) / 32;
    const unsigned *byn = blky + (size_t)n * NB;
    for (int bb0 = 0; bb0 < NB; bb0 += 32) {
        // 32 blocks at a time: which of them can reach this row at all?
        bool reach = false;
        if (bb0 + lane < NB) {
            const unsigned br = __ldg(byn + bb0 + lane);
            const int b0 = (int)(br & 0xffffu), b1 = (int)(br >> 16);
            reach = (b0 <= b1) && (b0 <= yhi) && (b1 >= ylo);
        }
        unsigned bm = __ballot_sync(0xffffffffu, reach);
        while (bm) {
            const int j = (bb0 + __ffs(bm) - 1) * 32 + lane;
            bm &= bm - 1;
            bool in = false;
            int k = 0;
            unsigned xr = 0;
            if (j < K) {
                k = slab_at_rank(ordn, K, kstart, j);
                const unsigned yr = __ldg(ryn + k);
                const int y0 = (int)(yr & 0xffffu), y1 = (int)(yr >> 16);
                in = (y0 <= y1) && (y0 <= yhi) && (y1 >= ylo);
                if (in) xr = __ldg(rxn + k);
            }
            const unsigned b = __ballot_sync(0xffffffffu, in);
            const int pos = total + __popc(b & below);
            if (in && pos < rowcap) { RowEntry e; e.k = k; e.xr = xr; out[pos] = e; }
            total += __popc(b);
        }
    }
    if (lane == 0) rowcnt[(size_t)n * R + row] = total;   // may exceed rowcap: consumers then scan all slabs
#if MVP_XBUCKETS
    // Second level: for every group of kGrpTiles tile columns, the row's entries (still in rank order) whose pixel range
    // touches the group, packed one group after the other into the row's group buffer (even offsets: 16-byte aligned for
    // the TMA staging).  Groups that no longer fit, and rows whose bucket overflowed, are marked (-1, -1): their tiles keep
    // scanning the row bucket.
    {
        __syncwarp();                          // this warp's bucket writes are visible to all its lanes
        int2 *hdr = grphdr + ((size_t)n * R + row) * NG;
        RowEntry *gout = grplist + ((size_t)n * R + row) * kGrpCap;
        int goff = 0;
        unsigned short *tc = tilecnt ? tilecnt + ((size_t)n * R + row) * TXn : nullptr;   // candidate slabs per tile: the cost estimate of order_ctas_kernel
        for (int g = 0; g < NG; ++g) {
            if (total > rowcap) {
                if (lane == 0) hdr[g] = make_int2(-1, -1);
                if (tilecnt && lane < kGrpTiles && g * kGrpTiles + lane < TXn) tc[g * kGrpTiles + lane] = 0xffff;
                continue;
            }
            const int gx0 = g * kGrpTiles * kTileW, gx1 = gx0 + kGrpTiles * kTileW - 1;
            int cnt = 0, mine = 0;
            for (int j0 = 0; j0 < total; j0 += 32) {
                const int j = j0 + lane;
                bool in = false;
                RowEntry e;
                e.k = 0; e.xr = 0;
                int x0 = 1, x1 = 0;
                if (j < total) {
                    e = out[j];
                    x0 = (int)(e.xr & 0xffffu); x1 = (int)(e.xr >> 16);
                    in = (x0 <= x1) && (x0 <= gx1) && (x1 >= gx0);
                }
                const unsigned b = __ballot_sync(0xffffffffu, in);
                const int pos = goff + cnt + __popc(b & below);
                if (in && pos < kGrpCap) gout[pos] = e;
                cnt += __popc(b);
                if (tilecnt) {
#pragma unroll
                    for (int t = 0; t < kGrpTiles; ++t) {
                        const int tx0 = gx0 + t * kTileW;
                        const unsigned bt = __ballot_sync(0xffffffffu, in && (x0 <= tx0 + kTileW - 1) && (x1 >= tx0));
                        if (lane == t) mine += __popc(bt);
                    }
                }
            }
            const bool ok = goff + cnt <= kGrpCap;
            if (lane == 0) hdr[g] = ok ? make_int2(goff, cnt) : make_int2(-1, -1);
            if (ok) goff += (cnt + 1) & ~1;
            if (tilecnt && lane < kGrpTiles && g * kGrpTiles + lane < TXn) tc[g * kGrpTiles + lane] = (unsigned short)min(mine, 0xffff);
        }
    }
#endif
}

// Same buckets, built by one CTA (8 warps) per (tile row, view): every warp owns a contiguous eighth of the rank-ordered slab
// sequence (count pass, prefix over the 8 warps, write pass) and a share of the x-groups.  A warp-per-row walk is a chain of
// ~630 dependent iterations -- 330 us however few views a launch has -- so this form is used for small launches (one rank of
// an 8-GPU run), where it is 5x shorter; large launches are throughput-bound and keep the single-pass kernel above.
__global__ void __launch_bounds__(kRowThreads) row_lists_cta_kernel(int K, int R, int rowcap, int TXn,
                                                                    const unsigned *__restrict__ rx, const unsigned *__restrict__ ry,
                                                                    const unsigned *__restrict__ blky, const int *__restrict__ order, int ostride,
                                                                    int *__restrict__ rowcnt, RowEntry *__restrict__ rowlist
#if MVP_XBUCKETS
                                                                    , int NG, int2 *__restrict__ grphdr, RowEntry *__restrict__ grplist,
                                                                    unsigned short *__restrict__ tilecnt
#endif
                                                                    ) {
    constexpr int NW = kRowThreads / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = blockIdx.x, n = blockIdx.y;
    const int ylo = row * kTileH, yhi = ylo + kTileH - 1;
    const unsigned *rxn = rx + (size_t)n * K, *ryn = ry + (size_t)n * K;
    RowEntry *out = rowlist + ((size_t)n * R + row) * rowcap;
    const int kstart = dfs_kstart(K);
    const int *ordn = order ? order + (size_t)n * ostride : nullptr;
    const unsigned below = (1u << lane) - 1u;
    __shared__ int s_cnt[NW];
    // the warp's segment of the rank-ordered sequence, in blocks of 32 slabs; only blocks whose y range reaches the row are read
    const int NB = (K + 31) / 32;
    const unsigned *byn = blky + (size_t)n * NB;
    const int bper = (NB + NW - 1) / NW;
    const int b_lo = warp * bper, b_hi = min(NB, b_lo + bper);
    auto test = [&](int j, int &k, bool &in) {
        in = false;
        k = 0;
        if (j < K) {
            k = slab_at_rank(ordn, K, kstart, j);
            const unsigned yr = __ldg(ryn + k);
            const int y0 = (int)(yr & 0xffffu), y1 = (int)(yr >> 16);
            in = (y0 <= y1) && (y0 <= yhi) && (y1 >= ylo);
        }
    };
    auto reach_mask = [&](int bb0) {
        bool reach = false;
        if (bb0 + lane < b_hi) {
            const unsigned br = __ldg(byn + bb0 + lane);
            const int b0 = (int)(br & 0xffffu), b1 = (int)(br >> 16);
            reach = (b0 <= b1) && (b0 <= yhi) && (b1 >= ylo);
        }
        return __ballot_sync(0xffffffffu, reach);
    };
    int mine = 0;
    for (int bb0 = b_lo; bb0 < b_hi; bb0 += 32) {
        unsigned bm = reach_mask(bb0);
        while (bm) {
            int k; bool in;
            test((bb0 + __ffs(bm) - 1) * 32 + lane, k, in);
            bm &= bm - 1;
            mine += __popc(__ballot_sync(0xffffffffu, in));
        }
    }
    if (lane == 0) s_cnt[warp] = mine;
    __syncthreads();
    int base = 0, total = 0;
    for (int w = 0; w < NW; ++w) { if (w < warp) base += s_cnt[w]; total += s_cnt[w]; }
    for (int bb0 = b_lo; bb0 < b_hi; bb0 += 32) {
        unsigned bm = reach_mask(bb0);
        while (bm) {
            int k; bool in;
            test((bb0 + __ffs(bm) - 1) * 32 + lane, k, in);
            bm &= bm - 1;
            const unsigned b = __ballot_sync(0xffffffffu, in);
            const int pos = base + __popc(b & below);
            if (in && pos < rowcap) { RowEntry e; e.k = k; e.xr = __ldg(rxn + k); out[pos] = e; }
            base += __popc(b);
        }
    }
    if (threadIdx.x == 0) rowcnt[(size_t)n * R + row] = total;
#if MVP_XBUCKETS
    {
        __shared__ int s_gcnt[64];               // entries per x-group (NG <= 64 groups are parallelised; more: see below)
        __shared__ int s_goff[64];
        __threadfence_block();
        __syncthreads();                          // the row bucket is complete and visible to the whole CTA
        int2 *hdr = grphdr + ((size_t)n * R + row) * NG;
        RowEntry *gout = grplist + ((size_t)n * R + row) * kGrpCap;
        unsigned short *tc = tilecnt ? tilecnt + ((size_t)n * R + row) * TXn : nullptr;
        if (total > rowcap || NG > 64) {
            // overflowed row (its tiles scan all slabs), or an image wider than 64 groups (4096 pixels): no second level
            for (int g = threadIdx.x; g < NG; g += kRowThreads) hdr[g] = make_int2(-1, -1);
            if (tc) for (int t = threadIdx.x; t < TXn; t += kRowThreads) tc[t] = 0xffff;
            return;
        }
        // count pass: warp w takes groups w, w + NW, ...
        for (int g = warp; g < NG; g += NW) {
            const int gx0 = g * kGrpTiles * kTileW, gx1 = gx0 + kGrpTiles * kTileW - 1;
            int cnt = 0, tmine = 0;
            for (int j0 = 0; j0 < total; j0 += 32) {
                const int j = j0 + lane;
                bool in = false;
                int x0 = 1, x1 = 0;
                if (j < total) {
                    const RowEntry e = out[j];
                    x0 = (int)(e.xr & 0xffffu); x1 = (int)(e.xr >> 16);
                    in = (x0 <= x1) && (x0 <= gx1) && (x1 >= gx0);
                }
                cnt += __popc(__ballot_sync(0xffffffffu, in));
                if (tc) {
#pragma unroll
                    for (int t = 0; t < kGrpTiles; ++t) {
                        const int tx0 = gx0 + t * kTileW;
                        const unsigned bt = __ballot_sync(0xffffffffu, in && (x0 <= tx0 + kTileW - 1) && (x1 >= tx0));
                        if (lane == t) tmine += __popc(bt);
                    }
                }
            }
            if (lane == 0) s_gcnt[g] = cnt;
            if (tc && lane < kGrpTiles && g * kGrpTiles + lane < TXn) tc[g * kGrpTiles + lane] = (unsigned short)min(tmine, 0xffff);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int goff = 0;
            for (int g = 0; g < NG; ++g) {
                const bool ok = goff + s_gcnt[g] <= kGrpCap;
                s_goff[g] = ok ? goff : -1;
                hdr[g] = ok ? make_int2(goff, s_gcnt[g]) : make_int2(-1, -1);
                if (ok) goff += (s_gcnt[g] + 1) & ~1;
            }
        }
        __syncthreads();
        // write pass
        for (int g = warp; g < NG; g += NW) {
            const int goff = s_goff[g];
            if (goff < 0) continue;
            const int gx0 = g * kGrpTiles * kTileW, gx1 = gx0 + kGrpTiles * kTileW - 1;
            int cnt = 0;
            for (int j0 = 0; j0 < total; j0 += 32) {
                const int j = j0 + lane;
                bool in = false;
                RowEntry e;
                e.k = 0; e.xr = 0;
                if (j < total) {
                    e = out[j];
                    const int x0 = (int)(e.xr & 0xffffu), x1 = (int)(e.xr >> 16);
                    in = (x0 <= x1) && (x0 <= gx1) && (x1 >= gx0);
                }
                const unsigned b = __ballot_sync(0xffffffffu, in);
                if (in) gout[goff + cnt + __popc(b & below)] = e;
                cnt += __popc(b);
            }
        }
    }
#endif
}

// ------------------------------------------------------------------------------------------------------
// 3b. CTA order: counting sort of the launch's CTAs (2x2 tiles) by descending cost class.  Cost estimate = the number of
//     candidate slabs of the CTA's four tiles (counted by row_lists_kernel), which correlates 0.72-0.76 with the measured
//     duration of a tile on B200 (scripts/tile_clocks.py).
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cta_cost_class(int n, int by, int bx, int R, int TXn, const unsigned short *__restrict__ tilecnt) {
    int cost = 0;
    for (int r = by * kBlkTY; r < min((by + 1) * kBlkTY, R); ++r)
        for (int t = bx * kBlkTX; t < min((bx + 1) * kBlkTX, TXn); ++t) cost += tilecnt[((size_t)n * R + r) * TXn + t];
    const int c = min(kCostClasses - 1, cost >> 3);
    return c >= MVP_CTA_ORDER_MIN ? c : 0;
}

// pass 0: histogram of the classes (hist[0 .. kCostClasses));  pass 1: scatter (cursor = hist[kCostClasses ..), zeroed).
// Both passes count in shared memory first and touch the global counters once per (block, class): the launch's CTAs fall into
// a handful of classes, so per-thread global atomics would serialise on a few addresses.
__global__ void __launch_bounds__(256) order_ctas_kernel(int pass, int N, int CXn, int CYn, int R, int TXn,
                                                         const unsigned short *__restrict__ tilecnt, int *__restrict__ hist,
                                                         int *__restrict__ order) {
    __shared__ int s_cnt[kCostClasses];
    __shared__ int s_base[kCostClasses];
    for (int c = threadIdx.x; c < kCostClasses; c += blockDim.x) s_cnt[c] = 0;
    __syncthreads();
    const size_t total = (size_t)N * CXn * CYn;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int c = 0, local = 0;
    if (i < total) {
        const int bx = (int)(i % CXn), by = (int)((i / CXn) % CYn), n = (int)(i / ((size_t)CXn * CYn));
        c = cta_cost_class(n, by, bx, R, TXn, tilecnt);
        local = atomicAdd(&s_cnt[c], 1);          // rank of this CTA among the block's CTAs of its class
    }
    __syncthreads();
    if (pass == 0) {
        for (int k = threadIdx.x; k < kCostClasses; k += blockDim.x)
            if (s_cnt[k]) atomicAdd(hist + k, s_cnt[k]);
        return;
    }
    // descending cost: class kCostClasses-1 first; the block reserves one range per class
    for (int k = threadIdx.x; k < kCostClasses; k += blockDim.x) {
        int before = 0;
        for (int q = kCostClasses - 1; q > k; --q) before += hist[q];
        s_base[k] = s_cnt[k] ? before + atomicAdd(hist + kCostClasses + k, s_cnt[k]) : 0;
    }
    __syncthreads();
    if (i < total) order[s_base[c] + local] = (int)i;
}

// ------------------------------------------------------------------------------------------------------
// device helpers shared by forward and backward
// ------------------------------------------------------------------------------------------------------
// bits of the lanes below this one (one special-register read; (1u << lane) - 1u is re-derived from %tid under a tight register cap)
__device__ __forceinline__ unsigned lanemask_lt() {
#ifdef MVP_CPU_EMUL
    return (1u << (threadIdx.x & 31)) - 1u;
#else
    unsigned m;
    asm volatile("mov.u32 %0, %%lanemask_lt;" : "=r"(m));   // volatile: read where it is used, not hoisted into a register that lives across the kernel
    return m;
#endif
}

// strictly inside the slab, |y_i| < 1 for all three (primsampler.h:46): the magnitudes compared as integers -- one 3-input maximum and one
// compare instead of three float compares and their predicate logic (forward event loop; with the constant slab size and lanemask_lt():
// -2.8 % instructions, -1 % time on B200).  Same decisions: below 1.0 the order of non-negative floats is the
// order of their bit patterns, a NaN's pattern is above 1.0's (invalid, as with the float compare), and flushing denormals changes nothing.
__device__ __forceinline__ bool inside_unit(float y0, float y1, float y2) {
    const unsigned a = __float_as_uint(y0) & 0x7fffffffu, b = __float_as_uint(y1) & 0x7fffffffu, c = __float_as_uint(y2) & 0x7fffffffu;
    return max(max(a, b), c) < 0x3f800000u;
}

struct Prim {
    float px, py, pz;
    float r00, r01, r02, r10, r11, r12, r20, r21, r22;
    float sx, sy, sz;
};

__device__ __forceinline__ Prim load_prim(const float4 *__restrict__ packn, int k) {
    const float4 *p = packn + (size_t)k * 4;
    float4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2), d = __ldg(p + 3);
    Prim q;
    q.px = a.x; q.py = a.y; q.pz = a.z; q.sx = a.w;
    q.r00 = b.x; q.r01 = b.y; q.r02 = b.z; q.sy = b.w;
    q.r10 = c.x; q.r11 = c.y; q.r12 = c.z; q.sz = c.w;
    q.r20 = d.x; q.r21 = d.y; q.r22 = d.z;
    return q;
}

// (v . R)_j as the reference compiles it: fma(R2j, v.z, fma(R0j, v.x, R1j * v.y))   (primtransf.h:128-131)
__device__ __forceinline__ float rowdot(float c0, float x, float c1, float y, float c2, float z) {
    return __fmaf_rn(c2, z, __fmaf_rn(c0, x, __fmul_rn(c1, y)));
}

struct Ray {
    float ox, oy, oz, dx, dy, dz, tmin, tmax;
};

// 1/x as the reference gets it under -use_fast_math (MUFU.RCP)
__device__ __forceinline__ float fast_rcp(float x) {
#ifdef MVP_CPU_EMUL
    return 1.f / x;
#else
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}

// utils.h:744-755: line vs slab in slab coordinates.  Returns hit; lo/hi valid when hit.
__device__ __forceinline__ bool slab_test(const Prim &q, const Ray &r, float &lo, float &hi) {
    float xm = r.ox - q.px, ym = r.oy - q.py, zm = r.oz - q.pz;
    float rx0 = rowdot(q.r00, xm, q.r10, ym, q.r20, zm), rd0 = rowdot(q.r00, r.dx, q.r10, r.dy, q.r20, r.dz);
    float rx1 = rowdot(q.r01, xm, q.r11, ym, q.r21, zm), rd1 = rowdot(q.r01, r.dx, q.r11, r.dy, q.r21, r.dz);
    float rx2 = rowdot(q.r02, xm, q.r12, ym, q.r22, zm), rd2 = rowdot(q.r02, r.dx, q.r12, r.dy, q.r22, r.dz);
    float i0 = fast_rcp(__fmul_rn(q.sx, rd0)), i1 = fast_rcp(__fmul_rn(q.sy, rd1)), i2 = fast_rcp(__fmul_rn(q.sz, rd2));
    float a0 = __fmul_rn(__fmaf_rn(q.sx, -rx0, -1.f), i0), b0 = __fmul_rn(__fmaf_rn(q.sx, -rx0, 1.f), i0);
    float a1 = __fmul_rn(__fmaf_rn(q.sy, -rx1, -1.f), i1), b1 = __fmul_rn(__fmaf_rn(q.sy, -rx1, 1.f), i1);
    float a2 = __fmul_rn(__fmaf_rn(q.sz, -rx2, -1.f), i2), b2 = __fmul_rn(__fmaf_rn(q.sz, -rx2, 1.f), i2);
    lo = fmaxf(fmaxf(fminf(a0, b0), fminf(a1, b1)), fminf(a2, b2));
    hi = fminf(fminf(fmaxf(a0, b0), fmaxf(a1, b1)), fmaxf(a2, b2));
    return lo <= hi;
}

#if MVP_LIST_MARGIN
// slab_test plus the interval [lom, him] of the same ray against the slab grown by `epos` (world units) on every side:
// per axis the crossing times move out by epos / |rd_i| = epos * |s_i * i_i|.
__device__ __forceinline__ bool slab_test_margin(const Prim &q, const Ray &r, float epos, float &lo, float &hi, float &lom, float &him) {
    float xm = r.ox - q.px, ym = r.oy - q.py, zm = r.oz - q.pz;
    float rx0 = rowdot(q.r00, xm, q.r10, ym, q.r20, zm), rd0 = rowdot(q.r00, r.dx, q.r10, r.dy, q.r20, r.dz);
    float rx1 = rowdot(q.r01, xm, q.r11, ym, q.r21, zm), rd1 = rowdot(q.r01, r.dx, q.r11, r.dy, q.r21, r.dz);
    float rx2 = rowdot(q.r02, xm, q.r12, ym, q.r22, zm), rd2 = rowdot(q.r02, r.dx, q.r12, r.dy, q.r22, r.dz);
    float i0 = fast_rcp(__fmul_rn(q.sx, rd0)), i1 = fast_rcp(__fmul_rn(q.sy, rd1)), i2 = fast_rcp(__fmul_rn(q.sz, rd2));
    float a0 = __fmul_rn(__fmaf_rn(q.sx, -rx0, -1.f), i0), b0 = __fmul_rn(__fmaf_rn(q.sx, -rx0, 1.f), i0);
    float a1 = __fmul_rn(__fmaf_rn(q.sy, -rx1, -1.f), i1), b1 = __fmul_rn(__fmaf_rn(q.sy, -rx1, 1.f), i1);
    float a2 = __fmul_rn(__fmaf_rn(q.sz, -rx2, -1.f), i2), b2 = __fmul_rn(__fmaf_rn(q.sz, -rx2, 1.f), i2);
    const float n0 = fminf(a0, b0), x0 = fmaxf(a0, b0), n1 = fminf(a1, b1), x1 = fmaxf(a1, b1), n2 = fminf(a2, b2), x2 = fmaxf(a2, b2);
    lo = fmaxf(fmaxf(n0, n1), n2);
    hi = fminf(fminf(x0, x1), x2);
    // s_i = 0 (infinite slab along that axis) gives i_i = inf and s_i * i_i = NaN: fminf drops the NaN, the margin becomes
    // huge and the (already infinite) axis interval stays infinite
    const float w0 = epos * fminf(fabsf(q.sx * i0), 1e30f), w1 = epos * fminf(fabsf(q.sy * i1), 1e30f), w2 = epos * fminf(fabsf(q.sz * i2), 1e30f);
    lom = fmaxf(fmaxf(n0 - w0, n1 - w1), n2 - w2);
    him = fminf(fminf(x0 + w0, x1 + w1), x2 + w2);
    return lo <= hi;
}
#endif

__device__ __forceinline__ int clamp_step(float v) {   // float -> step index, saturating, NaN -> +big
    if (!(v == v)) return kBig;
    return (int)fminf(fmaxf(v, -(float)kBig), (float)kBig);
}

// warp step interval of a list entry, packed as two int16 (lo | hi << 16); the extreme values mean "unbounded", so
// clamping an interval that does not fit only ever widens it (a superset of active steps is always correct)
__device__ __forceinline__ int pack_iv(int lo, int hi) {
    lo = max(min(lo, 32767), -32768); hi = max(min(hi, 32767), -32768);
    return (lo & 0xffff) | (hi << 16);
}
__device__ __forceinline__ int iv_lo(int v) { const int l = (int)(short)(v & 0xffff); return l == -32768 ? -kBig : l; }
__device__ __forceinline__ int iv_hi(int v) { const int h = v >> 16; return h == 32767 ? kBig : h; }

// ---- TMA bulk copy (cp.async.bulk, global -> shared) + mbarrier, used to stage the tile row's bucket ----
constexpr int kStage = 32;   // bucket entries per staged chunk (256 B), double buffered per warp

#ifdef MVP_CPU_EMUL
// emulation: the bulk copy is a memcpy by the issuing lane; the mbarrier is a phase counter (try_wait.parity(P) succeeds
// once the phase of parity P has completed)
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int) { *bar = 0; }
__device__ __forceinline__ void mbar_fence_init() {}
__device__ __forceinline__ void mbar_inval(unsigned long long *) {}
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    memcpy(dst, src, bytes);
    *bar += 1;
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    while ((unsigned)(*(volatile unsigned long long *)bar & 1) == parity) emul::yield();
}
#else
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// Make the (generic-proxy) mbarrier initialisation visible to the async proxy of this CTA.  Deliberately NOT
// fence.mbarrier_init.release.cluster: a cluster-scope fence compiles to CCTL.IVALL, which invalidates the SM's whole
// L1D -- fatal for a kernel that lives off L1 hits and starts a new tile per warp all the time.
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// An mbarrier must be invalidated before its memory is initialised again (a persistent warp builds one list per tile;
// mbarrier.init on a live barrier is undefined -- on B200 it ends in "unspecified launch failure").
__device__ __forceinline__ void mbar_inval(unsigned long long *bar) {
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}
#endif

// This lane's ray: read from the caller's ray tensors, or -- mvp_camera -- generated from the view's camera record with the arithmetic
// of mvp_compute_raydirs (raygen.h; utils_kernel.cu:32-46), in which case raypos / raydir / tminmax are never touched.
__device__ __forceinline__ Ray fetch_ray(const float *__restrict__ raypos, const float *__restrict__ raydir, const float *__restrict__ tminmax,
                                         const float4 *__restrict__ raycam, int n, size_t r, int cx, int cy) {
    Ray ray;
    if (raycam) {
        const float4 q0 = __ldg(raycam + (size_t)n * 4), q1 = __ldg(raycam + (size_t)n * 4 + 1), q2 = __ldg(raycam + (size_t)n * 4 + 2),
                     q3 = __ldg(raycam + (size_t)n * 4 + 3);
        MvpRayCam c;
        c.ox = q0.x; c.oy = q0.y; c.oz = q0.z;
        c.R[0] = q0.w; c.R[1] = q1.x; c.R[2] = q1.y; c.R[3] = q1.z; c.R[4] = q1.w; c.R[5] = q2.x; c.R[6] = q2.y; c.R[7] = q2.z; c.R[8] = q2.w;
        c.pcx = q3.x; c.pcy = q3.y; c.fx = q3.z; c.fy = q3.w;
        ray.ox = c.ox; ray.oy = c.oy; ray.oz = c.oz;
        mvp_gen_ray(c, (float)cx, (float)cy, ray.dx, ray.dy, ray.dz, ray.tmin, ray.tmax);
    } else {
        ray.ox = __ldg(raypos + r * 3 + 0); ray.oy = __ldg(raypos + r * 3 + 1); ray.oz = __ldg(raypos + r * 3 + 2);
        ray.dx = __ldg(raydir + r * 3 + 0); ray.dy = __ldg(raydir + r * 3 + 1); ray.dz = __ldg(raydir + r * 3 + 2);
        const float2 tmm = __ldg(reinterpret_cast<const float2 *>(tminmax) + r);
        ray.tmin = tmm.x; ray.tmax = tmm.y;
    }
    return ray;
}

struct TileCtx {
    // per-lane
    Ray ray;
    bool inimg;
    float rt0, rt1;     // own-hit [lo, hi] union (rtminmax, utils.h:757-761)
    int off;            // lane step j = sweep m + off
    // warp
    int nl;             // list length
};

constexpr int kClearBufs = 5;
struct Params {
    int N, H, W, K, TD, TH, TW;
    int pview;                    // 1: primitive tensors are per view [N,K,...]; 0: one set [1,K,...] shared by all views
    float dt, fadescale, fadeexp;
    const float *raypos, *raydir, *tminmax;
    const float4 *raycam;         // per view 4 x float4 (raygen.h): the rays are generated from it instead of read (mvp_camera); or NULL
    const float *tplate;          // voxels of the kernels' TP: float4, or four bf16 (MVP_FLAG_TPLATE_BF16)
    const float4 *pack;
    const unsigned *rx, *ry;
    const int *rowcnt;
    const RowEntry *rowlist;
    int R, rowcap;
    int TXn, TYn;
    unsigned slab_bytes;          // TD*TH*TW*sizeof(voxel): 16 (fp32 payload) or 8 (bf16)
    const int *order, *rankof;    // explicit marching order (per view [K]) and its inverse, or NULL: the fixed-order rotation
    long long *tileclk;           // MVP_TILE_CLOCKS diagnostics
    int CXn, CYn;                 // CTAs (kBlkTX x kBlkTY tiles) per view in x / y
    int use_order;                // this launch follows ctaorder (else plain grid order)
    const int *ctaorder;          // CTA ids ((n * CYn + by) * CXn + bx) in descending order of estimated cost (MVP_CTA_ORDER)
    int *heavycnt;                // tiles whose slab list overflowed the fast kernel's shared-memory list in THIS call ...
    int *heavylist;               // ... and their ids ((n * TYn + ty) * TXn + tx), in no particular order; the 512-entry kernel renders them
#if MVP_XBUCKETS
    const int2 *grphdr;           // per (view, tile row, x-group): (offset into the row's group buffer, entries) or (-1, -1)
    const RowEntry *grplist;      // per (view, tile row): kGrpCap entries
    int NG;
#endif
#if MVP_LIST_REUSE
    int2 *tilehdr;                // per tile: (offset into the view's listbuf, entries) or (-1, -1) = not saved
    int2 *listbuf;                // per view `listcap` entries (slab index, packed step interval)
    int *listcur;                 // per view bump cursor
    int *rayj0;                   // per ray: first lattice step, or kNoHitJ0
    int listcap;                  // entries of storage per view (stride of listbuf)
    int listlimit;                // entries the forward may use (= listcap; smaller only under MVP_FLAG_TEST_TINY_LISTS)
#endif
    // forward outputs
    float *rayrgba, *raysat;
    int4 *rayaux;
    float *rgb_nchw, *alpha_nchw;          // optional image-plane outputs [N,3,H,W] / [N,1,H,W]
    // backward
    const float *grad_rayrgba;
    const float *g_rgb_nchw, *g_alpha_nchw;   // the gradient as image planes (when grad_rayrgba is NULL)
    const float *raysat_in;
    const int4 *rayaux_in;
    float *g_primpos, *g_primrot, *g_primscale, *g_tplate;
    // algo 1: warp field [N,K,WD,WH,WW,3] (primsampler.h:53-58) and its gradient
    const float *warp;
    float *g_warp;
    int WD, WH, WW;
    // gradient buffers the gradient-mode forward zero-fills for the coming backward (mvp_forward_args::clear_grad_*): base (or NULL),
    // floats, and float4s per warp of the fast render launch
    float *clr[kClearBufs];
    unsigned long long clrn[kClearBufs], clrper[kClearBufs];
};

#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
long long g_emul_list_chunks;   // 32-entry bucket chunks scanned by build_tile_list (forward + backward)
long long g_emul_bwd_stats[8];  // see render_backward_kernel
#endif

// No slab rectangle reaches this tile (three quarters of the tiles of a head-and-shoulders view): its rays hit nothing, whatever they
// are -- the render kernels neither read nor generate them.
__device__ __forceinline__ bool tile_bucket_empty(const Params &p, int n, int tx, int ty) {
    const int cnt = p.rowcnt[(size_t)n * p.R + ty];
    if (cnt > p.rowcap) return false;          // overflowed row bucket: the tile scans all slabs
#if MVP_XBUCKETS
    const int2 gh = __ldg(p.grphdr + ((size_t)n * p.R + ty) * p.NG + tx / kGrpTiles);
    if (gh.y >= 0) return gh.y == 0;
#endif
    return cnt == 0;
}

// Builds the warp's slab list (rank order, at most CAP entries in shared memory), each slab's warp step interval and
// each lane's rtminmax, in one pass over the tile row's bucket.
//
// Lane <-> sweep alignment: lane step j = sweep m + off with off = ceil((tref - tmin) / dt), tref = min tmin of the
// tile, i.e. all lanes of a tile are at (nearly) the same depth t at the same sweep step.  Lanes only ever wait (sweep
// steps before their own first step are idle), so any alignment reproduces the reference; measured on B200, equal
// depth beats both "every lane starts at its own first hit" (the reference's lock-step loop) and a plane fitted to
// the first-hit depths (0.57 vs 0.70 ms per 1024x667 view) because neighbouring slabs sit at randomly different
// depths while the sweep planes stay coherent.
// Returns false when the list would exceed CAP (< 512): the caller hands the tile to the 512-entry kernel.
template <int CAP, bool kPrefetch, typename TP>
__device__ __forceinline__ bool build_tile_list(const Params &p, float rdt, int n, int tx, int ty, int lane, TileCtx &c,
                                                int *s_k, int *s_iv, RowEntry *s_stage, unsigned long long *s_bar, float &t,
                                                float &x, float &y, float &z, float &r1e, int &j0) {
    const int px = tx * kTileW + (lane & 7), py = ty * kTileH + (lane >> 3);
    c.inimg = (px < p.W) && (py < p.H);
    const int cx = min(px, p.W - 1), cy = min(py, p.H - 1);
    const size_t r = ((size_t)n * p.H + cy) * p.W + cx;
    c.ray = fetch_ray(p.raypos, p.raydir, p.tminmax, p.raycam, n, r, cx, cy);
    c.rt0 = CUDART_INF_F; c.rt1 = -CUDART_INF_F;

    const float tsteps = c.ray.tmin * rdt;            // lattice origin of this lane, in steps
    float tref = c.inimg ? tsteps : CUDART_INF_F;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tref = fminf(tref, __shfl_xor_sync(0xffffffffu, tref, o));
    c.off = clamp_step(ceilf(tref - tsteps));
    const float foff = (float)c.off;
#if MVP_LIST_MARGIN
    // Bound on |computed position at step j - exact point o + (tmin + j dt) d| for every step of this ray: one rounding of at
    // most 2^-23 per component and step (|x| < 2), three more at the start, sqrt(3) for the norm; 2^-19 on top covers
    // the rounding inside the slab transform and the slab test themselves.  In steps: see eps0.
    const float nsteps = fmaxf(c.ray.tmax - c.ray.tmin, 0.f) * rdt + 8.f;
    const float epos = 1.7320508f * nsteps * 1.1920929e-7f + 1.9073486e-6f;
    const float eps0 = fmaxf(0.001953125f, nsteps * 4.7683716e-7f);
#endif

    const float4 *packn = p.pack + (size_t)(n * p.pview) * p.K * 4;
    const int cnt = p.rowcnt[(size_t)n * p.R + ty];
    const bool overflow = cnt > p.rowcap;
#if MVP_XBUCKETS
    int total = overflow ? p.K : cnt;
    const RowEntry *rl = p.rowlist + ((size_t)n * p.R + ty) * p.rowcap;
    if (!overflow) {
        const int2 gh = __ldg(p.grphdr + ((size_t)n * p.R + ty) * p.NG + tx / kGrpTiles);
        if (gh.y >= 0) { rl = p.grplist + ((size_t)n * p.R + ty) * kGrpCap + gh.x; total = gh.y; }
    }
#else
    const int total = overflow ? p.K : cnt;
    const RowEntry *rl = p.rowlist + ((size_t)n * p.R + ty) * p.rowcap;
#endif
    const unsigned *rxn = p.rx + (size_t)n * p.K, *ryn = p.ry + (size_t)n * p.K;
    const int tx0 = tx * kTileW, tx1 = tx0 + kTileW - 1, ty0 = ty * kTileH, ty1 = ty0 + kTileH - 1;
    const int kstart = dfs_kstart(p.K);
    int nl = 0;
    // The bucket is streamed through shared memory by the TMA engine in 256-byte chunks, double buffered: chunk c+1 is
    // in flight while the (long) exact slab tests of chunk c run, so the bucket's load latency is never exposed.
    auto stage_issue = [&](int ch) {
        if (lane == 0) {
            const int cntc = min(kStage, total - ch * kStage);
            tma_load_1d(s_stage + (ch & 1) * kStage, rl + (size_t)ch * kStage, (unsigned)(((cntc + 1) & ~1) * sizeof(RowEntry)), s_bar + (ch & 1));
        }
    };
    if (!overflow && total > 0) {
        if (lane == 0) { mbar_init(s_bar, 1); mbar_init(s_bar + 1, 1); mbar_fence_init(); }
        __syncwarp();
        stage_issue(0);
    }
    for (int base = 0; base < total; base += 32) {
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
        if (lane == 0) std::atomic_ref<long long>(g_emul_list_chunks).fetch_add(1);
#endif
        const int idx = base + lane;
        int k = 0;
        bool cand = false;
        const int ch = base / kStage;
        if (!overflow) {
            if (base + kStage < total) stage_issue(ch + 1);   // its buffer was last read two chunks ago (warp-synced since)
            mbar_wait(s_bar + (ch & 1), (unsigned)((ch >> 1) & 1));
        }
        if (idx < total) {
            unsigned xr;
            if (!overflow) {
                RowEntry e = s_stage[(ch & 1) * kStage + lane];
                k = e.k; xr = e.xr;
                cand = true;
            } else {
                k = slab_at_rank(p.order ? p.order + (size_t)(n * p.pview) * p.K : nullptr, p.K, kstart, idx);
                xr = __ldg(rxn + k);
                unsigned yr = __ldg(ryn + k);
                int y0 = (int)(yr & 0xffffu), y1 = (int)(yr >> 16);
                cand = (y0 <= y1) && (y0 <= ty1) && (y1 >= ty0);
            }
            int x0 = (int)(xr & 0xffffu), x1 = (int)(xr >> 16);
            cand = cand && (x0 <= x1) && (x0 <= tx1) && (x1 >= tx0);
        }
        unsigned m = __ballot_sync(0xffffffffu, cand);
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            const int kk = __shfl_sync(0xffffffffu, k, b);
            const Prim q = load_prim(packn, kk);
            float lo, hi;
#if MVP_LIST_MARGIN
            float lom, him;
            const bool hit = slab_test_margin(q, c.ray, epos, lo, hi, lom, him) && c.inimg;
#else
            const bool hit = slab_test(q, c.ray, lo, hi) && c.inimg;
#endif
            int jlo = kBig, jhi = -kBig;
#if MVP_LIST_MARGIN
            // steps at which this lane's COMPUTED position can be inside the slab: the exact-arithmetic interval of the slab
            // grown by the position-error bound, plus eps0 steps for the rounding of the t -> step conversion.  Lanes that
            // miss the slab by less than the bound contribute too (list membership and rtminmax stay the reference's).
            if (c.inimg && lom <= him) {
                jlo = clamp_step(ceilf(lom * rdt - tsteps - eps0) - foff);
                jhi = clamp_step(floorf(him * rdt - tsteps + eps0) - foff);
            }
#endif
            if (hit) {
                c.rt0 = fminf(c.rt0, lo); c.rt1 = fmaxf(c.rt1, hi);
                // lattice steps that can lie inside [lo, hi]: floor((lo-tmin)/dt) .. floor((hi-tmin)/dt) + 1 (one step of
                // slack on each side covers the fp difference between this quotient and the incremental t of the march)
#if !MVP_LIST_MARGIN
                jlo = clamp_step(floorf(lo * rdt - tsteps) - foff);
                jhi = clamp_step(floorf(hi * rdt - tsteps) + 1.f - foff);
#endif
            }
            if (__any_sync(0xffffffffu, hit)) {
                const int wlo = __reduce_min_sync(0xffffffffu, jlo), whi = __reduce_max_sync(0xffffffffu, jhi);
                if (nl < CAP) {
                    if (lane == 0) {
                        s_k[nl] = kk; s_iv[nl] = pack_iv(wlo, whi);
                    }
                    ++nl;
                } else if (CAP < kMaxHit) {
                    // the list does not fit this kernel's shared-memory capacity (warp-uniform): the 512-entry kernel takes the
                    // tile.  A bulk copy of the next bucket chunk may still be in flight into this warp's staging buffer.
                    if (!overflow && base + kStage < total) mbar_wait(s_bar + ((ch + 1) & 1), (unsigned)(((ch + 1) >> 1) & 1));
                    __syncwarp();
                    if (!overflow && lane == 0) { mbar_inval(s_bar); mbar_inval(s_bar + 1); }
                    __syncwarp();
                    return false;
                }
            }
        }
        __syncwarp();   // every lane has consumed this chunk before its buffer is refilled
    }
    __syncwarp();
    if (!overflow && total > 0 && lane == 0) { mbar_inval(s_bar); mbar_inval(s_bar + 1); }   // all staged chunks have been waited for
    c.nl = nl;
#if MVP_PREFETCH
    // TMA bulk prefetch (cp.async.bulk.prefetch.L2): pull the payload slabs this tile is about to sample into L2 while
    // the lattice set-up runs; one lane per slab, fire and forget.
    if (kPrefetch && p.slab_bytes >= 16) {
        const char *tp = reinterpret_cast<const char *>(p.tplate) + (size_t)(n * p.pview) * p.K * p.slab_bytes;
        for (int i = lane; i < nl; i += 32) {
            const char *a = tp + (size_t)s_k[i] * p.slab_bytes;
            if constexpr (sizeof(TP) == 16) {
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"(p.slab_bytes) : "memory");
            } else {
                // bf16 slabs are 8-byte aligned: the 16-byte granules that lie inside the slab (a hint, so the ends may go unfetched)
                const uintptr_t lo = ((uintptr_t)a + 15) & ~(uintptr_t)15, hi = ((uintptr_t)a + p.slab_bytes) & ~(uintptr_t)15;
                if (hi > lo)
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(lo), "r"((unsigned)(hi - lo)) : "memory");
            }
        }
    }
#endif
    // lattice snap (mvpraymarch_subset_kernel.h:63-72 as compiled)
    const float r0 = fmaxf(c.rt0, c.ray.tmin), r1 = fminf(c.rt1, c.ray.tmax);
    const float xs = __fmaf_rn(c.ray.dx, c.ray.tmin, c.ray.ox), ys = __fmaf_rn(c.ray.dy, c.ray.tmin, c.ray.oy),
                zs = __fmaf_rn(c.ray.dz, c.ray.tmin, c.ray.oz);
    const int incs = __float2int_rd(__fmul_rn(__fadd_rn(r0, -c.ray.tmin), rdt));
    const float fi = (float)incs;
    t = __fmaf_rn(fi, p.dt, c.ray.tmin);
    x = __fmaf_rn(__fmul_rn(c.ray.dx, fi), p.dt, xs);
    y = __fmaf_rn(__fmul_rn(c.ray.dy, fi), p.dt, ys);
    z = __fmaf_rn(__fmul_rn(c.ray.dz, fi), p.dt, zs);
    r1e = __fadd_rn(r1, 9.9999997473787516356e-06f);
    j0 = incs;
    return true;
}

#if MVP_LIST_REUSE
constexpr int kNoHitJ0 = -0x7fffffff - 1;
#ifdef MVP_CPU_EMUL
int g_emul_saved_list_tiles[2];   // [0] tiles whose saved list the backward loaded, [1] tiles it rebuilt
#endif

// Forward (gradient mode): keep what build_tile_list produced for the backward.
__device__ __forceinline__ void save_tile_list(const Params &p, int n, int tx, int ty, int lane, const TileCtx &c, const int *s_k,
                                               const int *s_iv, size_t r, bool hashit, int j0) {
    const int nl = c.nl;
    int base = 0;
    if (lane == 0 && nl > 0) base = atomicAdd(p.listcur + n, nl);
    base = __shfl_sync(0xffffffffu, base, 0);
    const bool ok = base + nl <= p.listlimit;
    if (ok) {
        int2 *dst = p.listbuf + (size_t)n * p.listcap + base;
        for (int i = lane; i < nl; i += 32) dst[i] = make_int2(s_k[i], s_iv[i]);
    }
    if (lane == 0) p.tilehdr[((size_t)n * p.TYn + ty) * p.TXn + tx] = ok ? make_int2(base, nl) : make_int2(-1, -1);
    if (c.inimg) p.rayj0[r] = hashit ? j0 : kNoHitJ0;
}

// Backward: restore the outputs of build_tile_list the adjoint uses (ray, off, list, first step and its position) from
// what the forward saved.  Returns (warp-uniform) 1 = loaded, 0 = this tile's list was not saved (rebuild it), 2 = it was
// saved but is longer than this kernel's shared-memory list (the 512-entry kernel takes the tile).
template <int CAP>
__device__ __forceinline__ int load_saved_tile_list(const Params &p, float rdt, int n, int tx, int ty, int lane, TileCtx &c, int *s_k,
                                                     int *s_iv, float &x, float &y, float &z, int &j0) {
    const int2 hdr = __ldg(p.tilehdr + ((size_t)n * p.TYn + ty) * p.TXn + tx);
#ifdef MVP_CPU_EMUL
    if (lane == 0) atomicAdd(&g_emul_saved_list_tiles[hdr.y < 0 ? 1 : 0], 1);   // test hook: which path did the tile take
#endif
    if (hdr.y < 0) return 0;
    if (hdr.y > CAP) return 2;
    if (hdr.y == 0) { c.nl = 0; return 1; }   // nothing to march: the caller returns before it looks at anything else
    const int px = tx * kTileW + (lane & 7), py = ty * kTileH + (lane >> 3);
    c.inimg = (px < p.W) && (py < p.H);
    const int cx = min(px, p.W - 1), cy = min(py, p.H - 1);
    const size_t r = ((size_t)n * p.H + cy) * p.W + cx;
    c.ray = fetch_ray(p.raypos, p.raydir, p.tminmax, p.raycam, n, r, cx, cy);
    const float tsteps = c.ray.tmin * rdt;
    float tref = c.inimg ? tsteps : CUDART_INF_F;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tref = fminf(tref, __shfl_xor_sync(0xffffffffu, tref, o));
    c.off = clamp_step(ceilf(tref - tsteps));
    const int2 *src = p.listbuf + (size_t)n * p.listcap + hdr.x;
    for (int i = lane; i < hdr.y; i += 32) {
        const int2 e = __ldg(src + i);
        s_k[i] = e.x; s_iv[i] = e.y;
    }
    __syncwarp();
    c.nl = hdr.y;
    j0 = c.inimg ? __ldg(p.rayj0 + r) : kNoHitJ0;
    const bool hit = j0 != kNoHitJ0;
    c.rt0 = hit ? 0.f : 1.f; c.rt1 = hit ? 1.f : 0.f;   // the adjoint only asks whether rt0 <= rt1
    if (!hit) j0 = 0;
    // position of lattice step j0 (mvpraymarch_subset_kernel.h:63-72 as compiled; same expressions as build_tile_list)
    const float xs = __fmaf_rn(c.ray.dx, c.ray.tmin, c.ray.ox), ys = __fmaf_rn(c.ray.dy, c.ray.tmin, c.ray.oy),
                zs = __fmaf_rn(c.ray.dz, c.ray.tmin, c.ray.oz);
    const float fi = (float)j0;
    x = __fmaf_rn(__fmul_rn(c.ray.dx, fi), p.dt, xs);
    y = __fmaf_rn(__fmul_rn(c.ray.dy, fi), p.dt, ys);
    z = __fmaf_rn(__fmul_rn(c.ray.dz, fi), p.dt, zs);
    return 1;
}
#endif

// One payload voxel (RGBA) of `tplate` as fp32.  The render kernels take the voxel type TP as a template parameter: float4, or
// uint2 holding four bfloat16 (MVP_FLAG_TPLATE_BF16; R in the low half of .x).  A bfloat16 is the top half of the float with the
// same value, so the conversion is exact and everything after the load is the fp32 kernel's arithmetic.
__device__ __forceinline__ float4 load_voxel(const float4 *v) { return __ldg(v); }
__device__ __forceinline__ float4 load_voxel(const uint2 *v) {
    const uint2 u = __ldg(v);
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xffff0000u));
}

// primsampler.h:44-66 + utils.h:408-502.  T > 0: cubic slab with compile-time strides; T == 0: runtime dims.
// Only called for valid samples (|y| < 1), for which (a) the reference's +-100 clamp is a no-op and (b) the only
// corner that can fall outside the slab is ix+1 == TW when fx rounds to exactly TW-1, with weight exactly 0.  The
// cell is clamped to TW-2 instead and the fractions are taken against the clamped cell: identical products in all
// other cases (fx - ix and (ix+1) - fx are the reference's expressions), weights (1, 0) in the edge case.
template <int T, typename TP>
__device__ __forceinline__ float4 sample_slab(const TP *__restrict__ slab, float y0, float y1, float y2, int TD, int TH, int TW,
                                              float fadescale, float fadeexp) {
    const int td = T > 0 ? T : TD, th = T > 0 ? T : TH, tw = T > 0 ? T : TW;
    const float fade = __expf(-fadescale * (__powf(fabsf(y0), fadeexp) + __powf(fabsf(y1), fadeexp) + __powf(fabsf(y2), fadeexp)));
    const float fx = ((y0 + 1.f) * 0.5f) * (float)(tw - 1);
    const float fy = ((y1 + 1.f) * 0.5f) * (float)(th - 1);
    const float fz = ((y2 + 1.f) * 0.5f) * (float)(td - 1);
    const int ix = __float2int_rd(fx), iy = __float2int_rd(fy), iz = __float2int_rd(fz);
    int cx, cy, cz;
    if (T >= 2) { cx = min(ix, T - 2); cy = min(iy, T - 2); cz = min(iz, T - 2); }
    else { cx = max(min(ix, tw - 2), 0); cy = max(min(iy, th - 2), 0); cz = max(min(iz, td - 2), 0); }
    const float bx0 = fx - (float)cx, bx1 = (float)(cx + 1) - fx;
    const float by0 = fy - (float)cy, by1 = (float)(cy + 1) - fy;
    const float bz0 = fz - (float)cz, bz1 = (float)(cz + 1) - fz;
    const int sx = tw > 1 ? 1 : 0, sy = th > 1 ? tw : 0, sz = td > 1 ? th * tw : 0;
    const int base = (cz * th + cy) * tw + cx;
    const TP *pc = slab + base;
    const float4 v000 = load_voxel(pc), v001 = load_voxel(pc + sx), v010 = load_voxel(pc + sy), v011 = load_voxel(pc + sy + sx);
    const float4 v100 = load_voxel(pc + sz), v101 = load_voxel(pc + sz + sx), v110 = load_voxel(pc + sz + sy), v111 = load_voxel(pc + sz + sy + sx);
    // (wx * wy) * wz, left-associated like the reference; corner order tnw,tne,tsw,tse,bnw,bne,bsw,bse
    const float w00 = bx1 * by1, w01 = bx0 * by1, w10 = bx1 * by0, w11 = bx0 * by0;
    float4 acc;
    float w;
    w = w00 * bz1; acc.x = w * v000.x; acc.y = w * v000.y; acc.z = w * v000.z; acc.w = w * v000.w;
    w = w01 * bz1; acc.x = __fmaf_rn(w, v001.x, acc.x); acc.y = __fmaf_rn(w, v001.y, acc.y); acc.z = __fmaf_rn(w, v001.z, acc.z); acc.w = __fmaf_rn(w, v001.w, acc.w);
    w = w10 * bz1; acc.x = __fmaf_rn(w, v010.x, acc.x); acc.y = __fmaf_rn(w, v010.y, acc.y); acc.z = __fmaf_rn(w, v010.z, acc.z); acc.w = __fmaf_rn(w, v010.w, acc.w);
    w = w11 * bz1; acc.x = __fmaf_rn(w, v011.x, acc.x); acc.y = __fmaf_rn(w, v011.y, acc.y); acc.z = __fmaf_rn(w, v011.z, acc.z); acc.w = __fmaf_rn(w, v011.w, acc.w);
    w = w00 * bz0; acc.x = __fmaf_rn(w, v100.x, acc.x); acc.y = __fmaf_rn(w, v100.y, acc.y); acc.z = __fmaf_rn(w, v100.z, acc.z); acc.w = __fmaf_rn(w, v100.w, acc.w);
    w = w01 * bz0; acc.x = __fmaf_rn(w, v101.x, acc.x); acc.y = __fmaf_rn(w, v101.y, acc.y); acc.z = __fmaf_rn(w, v101.z, acc.z); acc.w = __fmaf_rn(w, v101.w, acc.w);
    w = w10 * bz0; acc.x = __fmaf_rn(w, v110.x, acc.x); acc.y = __fmaf_rn(w, v110.y, acc.y); acc.z = __fmaf_rn(w, v110.z, acc.z); acc.w = __fmaf_rn(w, v110.w, acc.w);
    w = w11 * bz0; acc.x = __fmaf_rn(w, v111.x, acc.x); acc.y = __fmaf_rn(w, v111.y, acc.y); acc.z = __fmaf_rn(w, v111.z, acc.z); acc.w = __fmaf_rn(w, v111.w, acc.w);
    acc.w *= fade;
    return acc;
}


// ---- generic trilinear cell for an ARBITRARY position (utils.h:408-502: +-100 clamp, corners outside the grid
//      contribute nothing); used by the warp-field path (algo 1), where the warped position may leave the slab ----
struct CellG {
    int idx[8];        // voxel index of each corner, -1 if outside
    float w[8];        // trilinear weight of each corner
    float x0, x1, y0, y1, z0, z1;
};
__device__ __forceinline__ CellG cell_generic(float a0, float a1, float a2, int D, int H, int W) {
    CellG c;
    const float fx = fmaxf(-100.f, fminf(100.f, (a0 + 1.f) * 0.5f)) * (float)(W - 1);
    const float fy = fmaxf(-100.f, fminf(100.f, (a1 + 1.f) * 0.5f)) * (float)(H - 1);
    const float fz = fmaxf(-100.f, fminf(100.f, (a2 + 1.f) * 0.5f)) * (float)(D - 1);
    const int ix = __float2int_rd(fx), iy = __float2int_rd(fy), iz = __float2int_rd(fz);
    c.x0 = fx - (float)ix; c.x1 = (float)(ix + 1) - fx;
    c.y0 = fy - (float)iy; c.y1 = (float)(iy + 1) - fy;
    c.z0 = fz - (float)iz; c.z1 = (float)(iz + 1) - fz;
#pragma unroll
    for (int cn = 0; cn < 8; ++cn) {
        const int x = ix + (cn & 1), y = iy + ((cn >> 1) & 1), z = iz + ((cn >> 2) & 1);
        const bool inb = (x >= 0) && (x < W) && (y >= 0) && (y < H) && (z >= 0) && (z < D);
        c.idx[cn] = inb ? (z * H + y) * W + x : -1;
        c.w[cn] = (((cn & 1) ? c.x0 : c.x1) * ((cn & 2) ? c.y0 : c.y1)) * ((cn & 4) ? c.z0 : c.z1);
    }
    return c;
}

// primsampler.h:44-66 with dowarp = true: fade from y, warp field sampled at y, payload sampled at the warped position
template <typename TP>
__device__ __forceinline__ float4 sample_slab_warped(const TP *__restrict__ slab, const float *__restrict__ wk, float y0, float y1,
                                                     float y2, const Params &p) {
    const float fade = __expf(-p.fadescale * (__powf(fabsf(y0), p.fadeexp) + __powf(fabsf(y1), p.fadeexp) + __powf(fabsf(y2), p.fadeexp)));
    const CellG cw = cell_generic(y0, y1, y2, p.WD, p.WH, p.WW);
    float q0 = 0.f, q1 = 0.f, q2 = 0.f;
#pragma unroll
    for (int cn = 0; cn < 8; ++cn) {
        if (cw.idx[cn] >= 0) {
            const float *v = wk + (size_t)cw.idx[cn] * 3;
            q0 = __fmaf_rn(cw.w[cn], __ldg(v), q0); q1 = __fmaf_rn(cw.w[cn], __ldg(v + 1), q1); q2 = __fmaf_rn(cw.w[cn], __ldg(v + 2), q2);
        }
    }
    const CellG ct = cell_generic(q0, q1, q2, p.TD, p.TH, p.TW);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int cn = 0; cn < 8; ++cn) {
        if (ct.idx[cn] >= 0) {
            const float4 v = load_voxel(slab + ct.idx[cn]);
            acc.x = __fmaf_rn(ct.w[cn], v.x, acc.x); acc.y = __fmaf_rn(ct.w[cn], v.y, acc.y);
            acc.z = __fmaf_rn(ct.w[cn], v.z, acc.z); acc.w = __fmaf_rn(ct.w[cn], v.w, acc.w);
        }
    }
    acc.w *= fade;
    return acc;
}

#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
// work counters of the emulated forward (tests / design studies only): [0] (step, 32-slot word) ballots, [1] (step, slab)
// events, [2] events with at least one valid lane, [3] valid lanes (= samples queued), [4] flushes, [5] tiles with a list,
// [6] events with a lane geometrically inside the slab (whether or not it still marches), [7] such lanes
long long g_emul_fwd_stats[8];
// second set: [0] sweep steps executed by the step loop, [1] steps run through by the skip loop, [2] events whose slab is the slab of the
// tile's previous event, [3] ballot words with two or more active slabs, [4] events in such words
long long g_emul_fwd_stats2[8];
#define MVP_STAT(i, v) do { if (lane == 0) stat_[i] += (v); } while (0)
#define MVP_STAT2(i, v) do { if (lane == 0) stat2_[i] += (v); } while (0)
#else
#define MVP_STAT(i, v) ((void)0)
#define MVP_STAT2(i, v) ((void)0)
#endif

template <int CAP, bool kGrad>
struct __align__(16) FwdWarpSmem {   // per-warp shared state of the forward kernel
#if MVP_SMEM_UNION
    union {
        float4 ring[kRing];            // sample queue of the march ...
        RowEntry stage[2 * kStage];    // ... bucket chunks while the list is built (every bulk copy has been waited for before the march starts)
    };
#else
    float4 ring[kRing];
    RowEntry stage[2 * kStage];
#endif
    unsigned long long bar[2];
    int k[CAP];
    int iv[CAP];
    float ra[kRing];
    int rm[kGrad ? kRing : 1];
};

// ------------------------------------------------------------------------------------------------------
// 4. forward.  CAP = shared-memory list capacity per warp.  The CAP < 512 variant handles every tile whose list
//    fits (almost all) with a small shared-memory footprint (more L1 for the voxel gathers) and flags the rest;
//    the CAP == 512 variant then renders only the flagged tiles.
// ------------------------------------------------------------------------------------------------------
template <int T, bool kGrad, int CAP, bool kWarp, typename TP>
__device__ __forceinline__ bool forward_tile(const Params &p, const int n, const int tx, const int ty, const int lane, FwdWarpSmem<CAP, kGrad> *const S) {
    // all per-warp shared state lives in one record: every address below is (one pinned per-warp base) + immediate
    int *const sk = S->k, *const siv = S->iv, *const rm = S->rm;
    RowEntry *const sstage = S->stage;
    unsigned long long *const sbar = S->bar;
    float4 *const ring = S->ring;
    float *const ra = S->ra;

    if (tile_bucket_empty(p, n, tx, ty)) {
        // background tile: what the general path below writes for rays without a hit, without touching the rays
        const int px = tx * kTileW + (lane & 7), py = ty * kTileH + (lane >> 3);
        const bool inimg = (px < p.W) && (py < p.H);
        const size_t r = ((size_t)n * p.H + min(py, p.H - 1)) * p.W + min(px, p.W - 1);
#if MVP_LIST_REUSE
        if (kGrad) {
            if (lane == 0) p.tilehdr[((size_t)n * p.TYn + ty) * p.TXn + tx] = make_int2(0, 0);
            if (inimg) p.rayj0[r] = kNoHitJ0;
        }
#endif
        if (inimg) {
            if (p.rayrgba) reinterpret_cast<float4 *>(p.rayrgba)[r] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.rgb_nchw) {
                const size_t plane = (size_t)p.H * p.W, pix = r - (size_t)n * plane;
                float *o = p.rgb_nchw + (size_t)n * 3 * plane + pix;
                o[0] = 0.f; o[plane] = 0.f; o[2 * plane] = 0.f;
                p.alpha_nchw[(size_t)n * plane + pix] = 0.f;
            }
            if (kGrad) {
                p.raysat[r * 3 + 0] = -1.f; p.raysat[r * 3 + 1] = -1.f; p.raysat[r * 3 + 2] = -1.f;
                p.rayaux[r] = make_int4(0x7fffffff, 0, 0, 0x7ffffffe);   // (no saturating sample, -, -, first step - 1 of a ray with no first step)
            }
        }
        return true;
    }
    const float rdt = fast_rcp(p.dt);   // MUFU.RCP(stepsize), as the reference (SASS 0x16c0)
    TileCtx c;
    float t, x, y, z, r1e;
    int j0;
    if (!build_tile_list<CAP, true, TP>(p, rdt, n, tx, ty, lane, c, sk, siv, sstage, sbar, t, x, y, z, r1e, j0)) return false;

    const int px = tx * kTileW + (lane & 7), py = ty * kTileH + (lane >> 3);
    const size_t r = ((size_t)n * p.H + min(py, p.H - 1)) * p.W + min(px, p.W - 1);

    const bool hashit = c.inimg && (c.rt0 <= c.rt1);
#if MVP_LIST_REUSE
    if (kGrad) save_tile_list(p, n, tx, ty, lane, c, sk, siv, r, hashit, j0);
#endif
    bool done = !hashit || (t > r1e);
    const int ms = done ? kBig : (j0 - c.off);   // sweep step at which this lane starts marching

    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float sat0 = -1.f, sat1 = -1.f, sat2 = -1.f;
    int jsat = 0x7fffffff, ranksat = 0, jlast = j0 - 1;
    float abefore = 0.f;
    bool sat = false;

    const int nl = c.nl;
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
    long long stat_[8] = {0, 0, 0, 0, 0, 0, 0, 0}, stat2_[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int prevk_ = -1;
    if (nl > 0) MVP_STAT(5, 1);
    if (nl > 128) MVP_STAT2(5, 1);      // list-length tail: [5] > 128, [6] > 160, [7] > 192 entries
    if (nl > 160) MVP_STAT2(6, 1);
    if (nl > 192) MVP_STAT2(7, 1);
#endif
    const int nwords = (nl + 31) >> 5;
    const float4 *packn = p.pack + (size_t)(n * p.pview) * p.K * 4;
    // voxels per slab: a compile-time constant for the cubic 8^3 / 16^3 specialisations, so that a slab's address is a shift and an add
    // wherever the register cap makes the compiler re-derive it (it was ~30 of the 159 instructions of a batch gather)
    const size_t slabsz = T > 0 ? (size_t)(T * T * T) : (size_t)p.TD * p.TH * p.TW;
    const TP *tpn = reinterpret_cast<const TP *>(p.tplate) + (size_t)(n * p.pview) * p.K * slabsz;
    const int kstart = dfs_kstart(p.K);
    {
        // pinned: under the register cap the compiler would otherwise re-materialise this base address per event
        unsigned long long pa = (unsigned long long)packn;
        asm volatile("" : "+l"(pa));
        packn = reinterpret_cast<const float4 *>(pa);
    }
    auto list_k = [&](int slot) { return sk[slot]; };

    // Sample compaction.  At one (step, slab) event only ~10 of the 32 rays of a tile are inside the slab, so the valid
    // samples are queued (sample coordinates + owner lane + list slot) and the expensive gather/interpolation runs on
    // full batches of 32 queued samples, one per lane, whichever ray they belong to.  The results go back through shared
    // memory and every ray composites ITS samples in queue order = (step, rank) order, so the arithmetic and its order
    // are exactly the reference's.  A ray that saturates only learns so at the next flush; what it queued in between is
    // sampled in vain and then ignored.  (Measured: neutral at 8^3 / K=16384, -15 % forward time at 16^3 / K=4096.)
    int qn = 0;
    unsigned ownlo = 0, ownhi = 0;   // queue positions (0..63) holding this lane's pending samples
#if MVP_FWD_RING
    int qhead = 0;                   // 0 or 32: the half of the ring the next flush takes (ownlo / ownhi belong to halves 0 / 1)
#else
    constexpr int qhead = 0;
#endif
    // primaccum.h:63-79 for this ray's samples among the sampled entries of the flushed half (bit b of `mine` = ring[qhead + b])
    auto composite = [&](unsigned mine) {
        while (mine) {
            const int b = qhead + __ffs(mine) - 1;
            mine &= mine - 1;
            if (!sat) {
                const float4 rr = ring[b];
                const float aw = ra[b];
                const float newa = __fmaf_rn(aw, p.dt, acc.w);
                const float contrib = __fadd_rn(fminf(newa, 1.f), -acc.w);
                if (newa >= 1.f) {
                    sat0 = rr.x; sat1 = rr.y; sat2 = rr.z;
                    sat = true;
                    if (kGrad) {
                        jsat = rm[b] + c.off;
                        ranksat = rank_of_slab(p.rankof ? p.rankof + (size_t)(n * p.pview) * p.K : nullptr, p.K, kstart, sk[(__float_as_int(rr.w) >> 5) & 1023]);
                        abefore = acc.w;
                    }
                }
                acc.x = __fmaf_rn(contrib, rr.x, acc.x); acc.y = __fmaf_rn(contrib, rr.y, acc.y);
                acc.z = __fmaf_rn(contrib, rr.z, acc.z); acc.w = __fadd_rn(acc.w, contrib);
            }
        }
    };
    auto flush = [&](int cnt) {
        MVP_STAT(4, 1);
        const bool act = lane < cnt;
        const float4 rec = ring[qhead + (act ? lane : 0)];
        float4 sres = make_float4(0.f, 0.f, 0.f, 0.f);
        if (act) {
            const int kk = sk[(__float_as_int(rec.w) >> 5) & 1023];
            if (kWarp) sres = sample_slab_warped(tpn + (size_t)kk * slabsz, p.warp + ((size_t)(n * p.pview) * p.K + kk) * ((size_t)p.WD * p.WH * p.WW * 3), rec.x, rec.y, rec.z, p);
            else sres = sample_slab<T, TP>(tpn + (size_t)kk * slabsz, rec.x, rec.y, rec.z, p.TD, p.TH, p.TW, p.fadescale, p.fadeexp);
        }
        __syncwarp();
        if (act) { ring[qhead + lane] = make_float4(sres.x, sres.y, sres.z, rec.w); ra[qhead + lane] = sres.w; }
        __syncwarp();
#if MVP_FWD_RING
        composite((qhead ? ownhi : ownlo) & (cnt >= 32 ? 0xffffffffu : ((1u << cnt) - 1u)));
        __syncwarp();                  // the half is free again before anything is queued into it
        if (qhead) ownhi = 0; else ownlo = 0;
        qhead ^= 32;
        qn -= cnt;
        if (sat) done = true;
    };
#else
        composite(ownlo & (cnt >= 32 ? 0xffffffffu : ((1u << cnt) - 1u)));
        __syncwarp();
        // move what is left of the queue to the front
        const int n2 = qn - cnt;
        float4 mv = make_float4(0.f, 0.f, 0.f, 0.f);
        int mvm = 0;
        if (lane < n2) { mv = ring[32 + lane]; if (kGrad) mvm = rm[32 + lane]; }
        __syncwarp();
        if (lane < n2) { ring[lane] = mv; if (kGrad) rm[lane] = mvm; }
        __syncwarp();
        ownlo = ownhi; ownhi = 0;
        qn = n2;
        if (sat) done = true;
    };
#endif

    const int mstart = __reduce_min_sync(0xffffffffu, ms);
    if (nl > 0 && mstart < kBig) {
        // each lane keeps the interval of list slots `lane` and `lane + 32` in registers (lists are rarely longer)
        int lo0 = kBig, hi0 = -kBig, lo1 = kBig, hi1 = -kBig;
        if (lane < nl) { const int v = siv[lane]; lo0 = iv_lo(v); hi0 = iv_hi(v); }
        if (lane + 32 < nl) { const int v = siv[lane + 32]; lo1 = iv_lo(v); hi1 = iv_hi(v); }
        for (int m = mstart;; ++m) {
            const bool on = !done && (m >= ms);
            bool anyslab = false;
            MVP_STAT2(0, 1);
            for (int w = 0; w < nwords; ++w) {
                bool a;
                if (w == 0) a = (lo0 <= m) && (m <= hi0);
                else if (w == 1) a = (lo1 <= m) && (m <= hi1);
                else {
                    const int slot = w * 32 + lane;
                    if (slot < nl) { const int v = siv[slot]; a = (iv_lo(v) <= m) && (m <= iv_hi(v)); } else a = false;
                }
                unsigned word = __ballot_sync(0xffffffffu, a);
                anyslab |= (word != 0);
                MVP_STAT(0, 1);
                if (__popc(word) >= 2) { MVP_STAT2(3, 1); MVP_STAT2(4, __popc(word)); }
                while (word) {
                    const int b = __ffs(word) - 1;
                    word &= word - 1;
                    MVP_STAT(1, 1);
                    const int k = list_k(w * 32 + b);
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
                    if (k == prevk_) MVP_STAT2(2, 1);
                    prevk_ = k;
#endif
                    const Prim q = load_prim(packn, k);
                    // primtransf.h:119-132
                    const float xm = x - q.px, ym = y - q.py, zm = z - q.pz;
                    const float y0 = __fmul_rn(q.sx, rowdot(q.r00, xm, q.r10, ym, q.r20, zm));
                    const float y1 = __fmul_rn(q.sy, rowdot(q.r01, xm, q.r11, ym, q.r21, zm));
                    const float y2 = __fmul_rn(q.sz, rowdot(q.r02, xm, q.r12, ym, q.r22, zm));
                    const bool valid = inside_unit(y0, y1, y2);
                    const bool want = valid && on && !sat && (t < r1e);
                    const unsigned vm = __ballot_sync(0xffffffffu, want);
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
                    { const unsigned gm = __ballot_sync(0xffffffffu, valid && c.inimg); MVP_STAT(6, gm != 0); MVP_STAT(7, __popc(gm)); }
#endif
                    if (vm) {
                        MVP_STAT(2, 1); MVP_STAT(3, __popc(vm));
                        if (want) {
                            const int pos = (qhead + qn + __popc(vm & lanemask_lt())) & (kRing - 1);
                            ring[pos] = make_float4(y0, y1, y2, __int_as_float(lane | ((w * 32 + b) << 5)));
                            if (kGrad) rm[pos] = m;
                            if (pos < 32) ownlo |= 1u << pos; else ownhi |= 1u << (pos - 32);
                        }
                        qn += __popc(vm);
                        __syncwarp();
                        if (qn >= 32) flush(32);
                    }
                }
            }
            if (on) {
                if (kGrad && (t < r1e)) jlast = m + c.off;
                t = __fadd_rn(t, p.dt);
                x = __fmaf_rn(c.ray.dx, p.dt, x); y = __fmaf_rn(c.ray.dy, p.dt, y); z = __fmaf_rn(c.ray.dz, p.dt, z);
                done = (t > r1e) || sat;
            }
            if (__all_sync(0xffffffffu, done)) break;
            if (!anyslab) {
                // nothing is active at this step: run ahead to the next step at which a slab becomes active, carrying
                // t and the position with the same per-step fma sequence (the result must not depend on the skipping)
                int nxt = kBig;
                if (lo0 > m) nxt = lo0;
                if (lo1 > m) nxt = min(nxt, lo1);
                for (int w = 2; w < nwords; ++w) {
                    const int slot = w * 32 + lane;
                    if (slot < nl) { const int l = iv_lo(siv[slot]); if (l > m) nxt = min(nxt, l); }
                }
                nxt = __reduce_min_sync(0xffffffffu, nxt);
                if (nxt == kBig) break;          // no slab starts later: nothing left to sample for any lane
                for (int mm = m + 1; mm < nxt; ++mm) {
                    MVP_STAT2(1, 1);
                    if (!done && (mm >= ms)) {
                        if (kGrad && (t < r1e)) jlast = mm + c.off;
                        t = __fadd_rn(t, p.dt);
                        x = __fmaf_rn(c.ray.dx, p.dt, x); y = __fmaf_rn(c.ray.dy, p.dt, y); z = __fmaf_rn(c.ray.dz, p.dt, z);
                        done = (t > r1e);
                    }
                }
                m = nxt - 1;
                if (__all_sync(0xffffffffu, done)) break;
            }
        }
    }
    if (qn > 0) flush(qn);
    if (c.inimg) {
        if (p.rayrgba) reinterpret_cast<float4 *>(p.rayrgba)[r] = acc;
        if (p.rgb_nchw) {
            // image planes for the caller (mvpraymarcher.py:50-51: permute + two contiguous copies, done here by the epilogue)
            const size_t plane = (size_t)p.H * p.W, pix = r - (size_t)n * plane;
            float *o = p.rgb_nchw + (size_t)n * 3 * plane + pix;
            o[0] = acc.x; o[plane] = acc.y; o[2 * plane] = acc.z;
            p.alpha_nchw[(size_t)n * plane + pix] = acc.w;
        }
        if (kGrad) {
            p.raysat[r * 3 + 0] = sat0; p.raysat[r * 3 + 1] = sat1; p.raysat[r * 3 + 2] = sat2;
            p.rayaux[r] = make_int4(jsat, ranksat, __float_as_int(abefore), jlast);
        }
    }
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
    if (lane == 0) for (int i = 0; i < 8; ++i) if (stat_[i]) std::atomic_ref<long long>(g_emul_fwd_stats[i]).fetch_add(stat_[i]);
    if (lane == 0) for (int i = 0; i < 8; ++i) if (stat2_[i]) std::atomic_ref<long long>(g_emul_fwd_stats2[i]).fetch_add(stat2_[i]);
#endif
    return true;
}

// Tiles whose slab list overflows the fast kernels' shared-memory list ("heavy" tiles: silhouette tiles of very dense
// scenes; none in the benchmark scene) are appended to a list by the fast kernel and rendered afterwards by the CAP == 512
// kernel, a small persistent grid that walks that list -- so the 512-entry launch costs a few microseconds when there is
// nothing to do, and the fast kernel's shared-memory footprint is set by the common case, not by the reference's cap.
constexpr int kHeavyGrid = 592;   // 4 CTAs per SM

template <int CAP, bool kGrad>
__device__ __forceinline__ FwdWarpSmem<CAP, kGrad> *pinned_warp_record(FwdWarpSmem<CAP, kGrad> *rec) {
#ifdef MVP_CPU_EMUL
    return rec;
#else
    unsigned woff = (unsigned)__cvta_generic_to_shared(rec);
    asm volatile("" : "+r"(woff));
    return reinterpret_cast<FwdWarpSmem<CAP, kGrad> *>(__cvta_shared_to_generic((size_t)woff));
#endif
}

// The gradient buffers of the coming backward, zero-filled on the side: warp g of the G warps of the fast render launch clears the g-th
// slice of each buffer with streaming 16-byte stores before it renders its tile.  The render kernel is issue bound with the DRAM
// write path idle, and 134 MB per view is 12 store instructions per warp -- a separate memset pass costs 1.4 ms per 80 views.
__device__ __forceinline__ void clear_grad_slices(const Params &p, size_t g, int lane) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int b = 0; b < kClearBufs; ++b) {
        float *const base = p.clr[b];
        if (!base) continue;
        const size_t n4 = p.clrn[b] >> 2, lo = g * p.clrper[b];
        const size_t hi = lo + p.clrper[b] < n4 ? lo + p.clrper[b] : n4;
        for (size_t i = lo + lane; i < hi; i += 32) __stcs(reinterpret_cast<float4 *>(base) + i, z);
        if (g == 0 && lane < (int)(p.clrn[b] & 3)) base[(n4 << 2) + lane] = 0.f;
    }
}

template <int T, bool kGrad, int CAP, bool kWarp, typename TP>
__global__ void __launch_bounds__(kWarps * 32, (CAP < kMaxHit && !kWarp) ? (MVP_FWD_MINB * 4) / kWarps : 16 / kWarps) render_forward_kernel(const Params p) {
    __shared__ FwdWarpSmem<CAP, kGrad> s_w[kWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    FwdWarpSmem<CAP, kGrad> *const S = pinned_warp_record<CAP, kGrad>(&s_w[warp]);
    // warps are independent: no CTA-wide barrier anywhere
    if (CAP == kMaxHit) {
        const int cnt = *p.heavycnt;
        for (int i = blockIdx.x * kWarps + warp; i < cnt; i += gridDim.x * kWarps) {
            const int id = p.heavylist[i];
            const int tx = id % p.TXn, ty = (id / p.TXn) % p.TYn, n = id / (p.TXn * p.TYn);
            forward_tile<T, kGrad, CAP, kWarp, TP>(p, n, tx, ty, lane, S);
            __syncwarp();
        }
    } else {
#if MVP_CTA_ORDER
        if (kGrad) clear_grad_slices(p, (size_t)blockIdx.x * kWarps + warp, lane);
        // 1-D grid; CTA b renders the b-th most expensive 2x2-tile block of the launch (order_ctas_kernel), or block b
        const int cid = p.use_order ? p.ctaorder[blockIdx.x] : (int)blockIdx.x;
        const int bx = cid % p.CXn, by = (cid / p.CXn) % p.CYn, n = cid / (p.CXn * p.CYn);
        const int tx = bx * kBlkTX + (warp % kBlkTX), ty = by * kBlkTY + (warp / kBlkTX);
#else
        const int tx = blockIdx.x * kBlkTX + (warp % kBlkTX), ty = blockIdx.y * kBlkTY + (warp / kBlkTX), n = blockIdx.z;
#endif
        if (tx >= p.TXn || ty >= p.TYn) return;
#if MVP_TILE_CLOCKS
        const long long t0_ = clock64();
        long long g0_;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0_));
#endif
        if (!forward_tile<T, kGrad, CAP, kWarp, TP>(p, n, tx, ty, lane, S) && lane == 0)
            p.heavylist[atomicAdd(p.heavycnt, 1)] = (n * p.TYn + ty) * p.TXn + tx;
#if MVP_TILE_CLOCKS
        if (lane == 0) {
            long long g1_;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1_));
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            long long *o = p.tileclk + (((size_t)n * p.TYn + ty) * p.TXn + tx) * 4;
            o[0] = g0_; o[1] = g1_; o[2] = clock64() - t0_; o[3] = (long long)smid | ((long long)blockIdx.x << 32);
        }
#endif
    }
}

// ------------------------------------------------------------------------------------------------------
// 5. backward (slab-major)
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void red_add_v4(float *addr, float a, float b, float c, float d) {
#ifdef MVP_EXPERIMENT_NO_RED   // timing experiment only: how much of the backward is the payload-gradient scatter?
    if (a == 12345.678f) addr[0] = b + c + d;
    return;
#endif
    // no "memory" clobber: the gradient buffer is never read in this kernel, loads must stay free to move
#ifdef MVP_CPU_EMUL
    atomicAdd(addr, a); atomicAdd(addr + 1, b); atomicAdd(addr + 2, c); atomicAdd(addr + 3, d);
#else
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d));
#endif
}

// dL/d(index) of one sample (utils.h:591-642) in full generality, i.e. including an axis whose cell was clamped (the sample sits
// exactly on the slab's far face: probability ~2^-24 per axis, the upper voxel is then the reference's LOWER corner and the only
// one it sees).  Taken by those samples only; it runs after the main corner pass, when few values of the batch adjoint are live, so its
// 12 accumulators do not add to the register peak.
template <typename TP>
__device__ __forceinline__ float3 index_grad_general(const TP *pc, int sx, int sy, int sz, float bx0, float bx1, float by0, float by1,
                                                  float bz0, float bz1, float oLx, float oLy, float oLz, float A, float B, int clamp_mask) {
    const float wx_[2] = {bx1, bx0}, wy_[2] = {by1, by0}, wz_[2] = {bz1, bz0};
    float gpU[3] = {0.f, 0.f, 0.f}, gpL[3] = {0.f, 0.f, 0.f}, gaU[3] = {0.f, 0.f, 0.f}, gaL[3] = {0.f, 0.f, 0.f};
    for (int cn = 0; cn < 8; ++cn) {
        const int bx = cn & 1, byy = (cn >> 1) & 1, bz = (cn >> 2) & 1;
        const float4 v = load_voxel(pc + ((bx ? sx : 0) + (byy ? sy : 0) + (bz ? sz : 0)));
        const float pr = v.x * oLx + v.y * oLy + v.z * oLz;
        const float wyz = wy_[byy] * wz_[bz], wxz = wx_[bx] * wz_[bz], wxy = wx_[bx] * wy_[byy];
        if (bx) { gpU[0] += pr * wyz; gaU[0] += v.w * wyz; } else { gpL[0] += pr * wyz; gaL[0] += v.w * wyz; }
        if (byy) { gpU[1] += pr * wxz; gaU[1] += v.w * wxz; } else { gpL[1] += pr * wxz; gaL[1] += v.w * wxz; }
        if (bz) { gpU[2] += pr * wxy; gaU[2] += v.w * wxy; } else { gpL[2] += pr * wxy; gaL[2] += v.w * wxy; }
    }
    float3 g;
    g.x = (clamp_mask & 1) ? -(A * gpU[0] + B * gaU[0]) : (A * (gpU[0] - gpL[0]) + B * (gaU[0] - gaL[0]));
    g.y = (clamp_mask & 2) ? -(A * gpU[1] + B * gaU[1]) : (A * (gpU[1] - gpL[1]) + B * (gaU[1] - gaL[1]));
    g.z = (clamp_mask & 4) ? -(A * gpU[2] + B * gaU[2]) : (A * (gpU[2] - gpL[2]) + B * (gaU[2] - gaL[2]));
    return g;
}

template <int CAP>
struct __align__(16) BwdWarpSmem {   // per-warp shared state of the backward kernel
#if MVP_SMEM_UNION
    union {
        float4 q[kRing];
        RowEntry stage[2 * kStage];    // only the list rebuild uses it, before the first sample is queued
    };
#else
    float4 q[kRing];
    RowEntry stage[2 * kStage];
#endif
    unsigned long long bar[2];
    int k[CAP];
    int iv[CAP];
    float ray[9 * 32];
    float4 rec[4];          // record of the slab being processed (MVP_BWD_SMEMREC)
#if MVP_BWD_LANESMEM
    float ls[24 * 32];      // [field][lane]: see backward_tile
#endif
};

// The slab record from shared memory through loads the compiler can neither hoist nor keep alive: the caller decides where the
// 15 values are live.
__device__ __forceinline__ Prim load_rec_shared(const float4 *rec) {
    float4 a, b, c, d;
#ifdef MVP_CPU_EMUL
    a = rec[0]; b = rec[1]; c = rec[2]; d = rec[3];
#else
    const unsigned addr = smem_u32(rec);
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(addr));
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+16];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(addr));
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+32];" : "=f"(c.x), "=f"(c.y), "=f"(c.z), "=f"(c.w) : "r"(addr));
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+48];" : "=f"(d.x), "=f"(d.y), "=f"(d.z), "=f"(d.w) : "r"(addr));
#endif
    Prim q;
    q.px = a.x; q.py = a.y; q.pz = a.z; q.sx = a.w;
    q.r00 = b.x; q.r01 = b.y; q.r02 = b.z; q.sy = b.w;
    q.r10 = c.x; q.r11 = c.y; q.r12 = c.z; q.sz = c.w;
    q.r20 = d.x; q.r21 = d.y; q.r22 = d.z;
    return q;
}

template <int T, int CAP, bool kWarp, typename TP>
__device__ __forceinline__ bool backward_tile(const Params &p, const int n, const int tx, const int ty, const int lane, BwdWarpSmem<CAP> *const S) {
    int *const sk = S->k, *const siv = S->iv;
    RowEntry *const sstage = S->stage;
    unsigned long long *const sbar = S->bar;
    float4 *const sq = S->q;
    float *const sray = S->ray;   // per-ray adjoint constants: dL.xyzw, saturation colour + flag, alpha before saturation

    const float rdt = fast_rcp(p.dt);
    TileCtx c;
    float t0, xb, yb, zb, r1e;   // xb = position at sweep step max(mcur, ms)
    int j0;
    int have = 0;           // 0: rebuild the list, 1: loaded what the forward saved, 2: the saved list does not fit this kernel
#if MVP_LIST_REUSE
    have = load_saved_tile_list<CAP>(p, rdt, n, tx, ty, lane, c, sk, siv, xb, yb, zb, j0);
    if (have == 2) return false;
#endif
    if (have == 0 && !build_tile_list<CAP, false, TP>(p, rdt, n, tx, ty, lane, c, sk, siv, sstage, sbar, t0, xb, yb, zb, r1e, j0)) return false;
    const int nl = c.nl;
    if (nl == 0) return true;

    const int px = tx * kTileW + (lane & 7), py = ty * kTileH + (lane >> 3);
    const size_t r = ((size_t)n * p.H + min(py, p.H - 1)) * p.W + min(px, p.W - 1);

    const bool hashit = c.inimg && (c.rt0 <= c.rt1);
    const int4 aux = __ldg(p.rayaux_in + r);
    const int msat = aux.x == 0x7fffffff ? 0x7fffffff : aux.x - c.off;   // in sweep units
    const int ranksat = aux.y;
    {
        // per-ray constants of the adjoint live in shared memory ([field][lane]: a batch reads them by owner lane,
        // conflict-free, instead of holding 9 registers per thread for the whole kernel)
        float4 dL;
        if (p.grad_rayrgba) dL = __ldg(reinterpret_cast<const float4 *>(p.grad_rayrgba) + r);
        else {
            const size_t plane = (size_t)p.H * p.W, pix = r - (size_t)n * plane;
            const float *gi = p.g_rgb_nchw + (size_t)n * 3 * plane + pix;
            dL = make_float4(__ldg(gi), __ldg(gi + plane), __ldg(gi + 2 * plane), __ldg(p.g_alpha_nchw + (size_t)n * plane + pix));
        }
        const float rs0 = __ldg(p.raysat_in + r * 3 + 0), rs1 = __ldg(p.raysat_in + r * 3 + 1), rs2 = __ldg(p.raysat_in + r * 3 + 2);
        const bool hassat = rs0 > -1.f;
        float *pr_ = sray;
        pr_[0 * 32 + lane] = dL.x; pr_[1 * 32 + lane] = dL.y; pr_[2 * 32 + lane] = dL.z; pr_[3 * 32 + lane] = dL.w;
        pr_[4 * 32 + lane] = hassat ? rs0 : 0.f; pr_[5 * 32 + lane] = hassat ? rs1 : 0.f; pr_[6 * 32 + lane] = hassat ? rs2 : 0.f;
        pr_[7 * 32 + lane] = hassat ? 1.f : 0.f;
        pr_[8 * 32 + lane] = __int_as_float(aux.z);      // alpha before the saturating sample
        __syncwarp();
    }

    // lane's live sweep range [ms, mlast]
    const int ms = hashit ? (j0 - c.off) : kBig;
    const int mlast = hashit ? (min(aux.w - c.off, msat)) : -1;
    const float foff = (float)c.off;
    const int wlast = __reduce_max_sync(0xffffffffu, mlast);
    const int wfirst = __reduce_min_sync(0xffffffffu, ms);
    if (wlast < wfirst || wfirst >= kBig) return true;

    const float4 *packn = p.pack + (size_t)(n * p.pview) * p.K * 4;
    const size_t slabsz = (size_t)p.TD * p.TH * p.TW;   // (a compile-time T^3 here makes the compiler keep slab addresses in registers: 64 B of spills)
    // bases of the primitive tensors are re-derived from the parameter block where they are used (cheap constant-bank
    // arithmetic) instead of living in a dozen registers for the whole tile
    const size_t pvK = (size_t)(n * p.pview) * p.K;
    const int td = T > 0 ? T : p.TD, th = T > 0 ? T : p.TH, tw = T > 0 ? T : p.TW;
    const float gmx = (float)(tw - 1) * 0.5f, gmy = (float)(th - 1) * 0.5f, gmz = (float)(td - 1) * 0.5f;
    const int sx = tw > 1 ? 1 : 0, sy = th > 1 ? tw : 0, sz = td > 1 ? th * tw : 0;
    const int kstart = dfs_kstart(p.K);

#if MVP_BWD_LANESMEM
    // per-lane state that is only read between batches: parked in shared memory ([field][lane], conflict-free), read back
    // through volatile accesses so that the compiler cannot keep it in registers across the batch adjoint
    volatile float *const ls = S->ls + lane;
    ls[0 * 32] = c.ray.ox; ls[1 * 32] = c.ray.oy; ls[2 * 32] = c.ray.oz; ls[3 * 32] = c.ray.tmin; ls[4 * 32] = c.ray.tmax;
    ls[5 * 32] = __int_as_float(ms); ls[6 * 32] = __int_as_float(mlast); ls[7 * 32] = __int_as_float(msat); ls[8 * 32] = __int_as_float(ranksat);
    ls[9 * 32] = xb; ls[10 * 32] = yb; ls[11 * 32] = zb;
#define L_OX ls[0 * 32]
#define L_OY ls[1 * 32]
#define L_OZ ls[2 * 32]
#define L_TMIN ls[3 * 32]
#define L_TMAX ls[4 * 32]
#define L_MS __float_as_int(ls[5 * 32])
#define L_MLAST __float_as_int(ls[6 * 32])
#define L_MSAT __float_as_int(ls[7 * 32])
#define L_RANKSAT __float_as_int(ls[8 * 32])
#define L_XB ls[9 * 32]
#define L_YB ls[10 * 32]
#define L_ZB ls[11 * 32]
#define L_GX(i) ls[(12 + (i)) * 32]
#else
#define L_OX c.ray.ox
#define L_OY c.ray.oy
#define L_OZ c.ray.oz
#define L_TMIN c.ray.tmin
#define L_TMAX c.ray.tmax
#define L_MS ms
#define L_MLAST mlast
#define L_MSAT msat
#define L_RANKSAT ranksat
#define L_XB xb
#define L_YB yb
#define L_ZB zb
#endif
    const float rdx = c.ray.dx, rdy = c.ray.dy, rdz = c.ray.dz;   // the only ray values the step loops need
    // Slabs are processed in the order of their first sweep step, 16-step chunk by chunk, so that each lane's
    // position can be carried forward with the SAME fma sequence the forward kernel executed (bit-identical sample
    // positions: the trilinear position gradient is discontinuous across voxel cells, so this matters).
    int mcur = wfirst;
    const int nwords = (nl + 31) >> 5;
    for (int cs = wfirst; cs <= wlast; cs += kMaskSteps) {
        if (mcur < cs) {
            float xb_ = L_XB, yb_ = L_YB, zb_ = L_ZB;
            const int ms_ = L_MS;
            for (; mcur < cs; ++mcur) {
                if (mcur >= ms_) { xb_ = __fmaf_rn(rdx, p.dt, xb_); yb_ = __fmaf_rn(rdy, p.dt, yb_); zb_ = __fmaf_rn(rdz, p.dt, zb_); }
            }
            L_XB = xb_; L_YB = yb_; L_ZB = zb_;
        }
        for (int w = 0; w < nwords; ++w) {
            const int myslot = w * 32 + lane;
            bool pick = false;
            if (myslot < nl) {
                const int v = siv[myslot];
                const int a0 = max(iv_lo(v), wfirst), b0 = min(iv_hi(v), wlast);
                pick = (a0 <= b0) && (a0 >= cs) && (a0 < cs + kMaskSteps);
            }
            unsigned word = __ballot_sync(0xffffffffu, pick);
            while (word) {
                const int bit = __ffs(word) - 1;
                word &= word - 1;
                const int slot = w * 32 + bit;
                const int k = sk[slot];
                const int rank = rank_of_slab(p.rankof ? p.rankof + (size_t)(n * p.pview) * p.K : nullptr, p.K, kstart, k);
#if MVP_BWD_SMEMREC
                __syncwarp();                                  // the previous slab's last readers of the record are done
                if (lane < 4) S->rec[lane] = __ldg(packn + (size_t)k * 4 + lane);
                __syncwarp();
#else
                const Prim q = load_prim(packn, k);
#endif
                // Slab-major order needs no cross-lane alignment: every lane walks ITS OWN step interval of this slab
                // (recomputed from the reference's slab test), so all rays that cross the slab are busy together.
                float lo, hi;
                int la = kBig, lb = -kBig;               // lane's candidate sweep steps [la, lb]
#if MVP_BWD_SMEMREC
                {
                const Prim q = load_rec_shared(S->rec);
#endif
#if MVP_LIST_MARGIN
                // same drift-bound intervals as the tile lists (build_tile_list); the bound is recomputed per slab instead
                // of living in two registers for the whole kernel
                {
                    Ray ry;
                    ry.ox = L_OX; ry.oy = L_OY; ry.oz = L_OZ; ry.dx = rdx; ry.dy = rdy; ry.dz = rdz; ry.tmin = L_TMIN; ry.tmax = L_TMAX;
                    const float nsteps = fmaxf(ry.tmax - ry.tmin, 0.f) * rdt + 8.f;
                    const float epos = 1.7320508f * nsteps * 1.1920929e-7f + 1.9073486e-6f;
                    const float eps0 = fmaxf(0.001953125f, nsteps * 4.7683716e-7f);
                    float lom, him;
                    slab_test_margin(q, ry, epos, lo, hi, lom, him);
                    if (hashit && lom <= him) {
                        la = max(clamp_step(ceilf((lom - ry.tmin) * rdt - eps0) - foff), max(L_MS, cs));
                        lb = min(clamp_step(floorf((him - ry.tmin) * rdt + eps0) - foff), L_MLAST);
                        if (rank > L_RANKSAT) lb = min(lb, L_MSAT - 1);      // samples after the saturating one do not exist
                    }
                }
                const bool hit = false;
#else
                Ray ry;
                ry.ox = L_OX; ry.oy = L_OY; ry.oz = L_OZ; ry.dx = rdx; ry.dy = rdy; ry.dz = rdz; ry.tmin = L_TMIN; ry.tmax = L_TMAX;
                const bool hit = slab_test(q, ry, lo, hi) && hashit;
#endif
                if (hit) {
                    // candidate lattice steps floor((lo-tmin)/dt) .. floor((hi-tmin)/dt)+1: the strictly-inside range plus one
                    // step of slack on each side, because lo/hi carry ~1e-6 relative error (rcp.approx) and the forward's
                    // validity test, not this interval, decides which samples exist.
                    la = max(clamp_step(floorf((lo - L_TMIN) * rdt) + MVP_BWD_LO_SLACK - foff), max(L_MS, cs));
                    lb = min(clamp_step(floorf((hi - L_TMIN) * rdt) + MVP_BWD_HI_SLACK - foff), L_MLAST);
                    if (rank > L_RANKSAT) lb = min(lb, L_MSAT - 1);      // samples after the saturating one do not exist
                }
#if MVP_BWD_SMEMREC
                }
#endif
                const int len = lb - la + 1;
                const int maxlen = __reduce_max_sync(0xffffffffu, len);
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
                // [0] (tile, slab) visits, [1] visits with work, [2] warp steps (sum of maxlen), [3] lane steps inside a lane's
                // interval, [4] valid lane steps (= samples), [5] batches, [6] position-carry steps
                if (lane == 0) { std::atomic_ref<long long>(g_emul_bwd_stats[0]).fetch_add(1); if (maxlen > 0) { std::atomic_ref<long long>(g_emul_bwd_stats[1]).fetch_add(1); std::atomic_ref<long long>(g_emul_bwd_stats[2]).fetch_add(maxlen); } }
                if (maxlen > 0 && len > 0) std::atomic_ref<long long>(g_emul_bwd_stats[3]).fetch_add(len);
#endif
                if (maxlen <= 0) continue;
                const TP *slab = reinterpret_cast<const TP *>(p.tplate) + (pvK + k) * slabsz;
                float *gslab = p.g_tplate + (pvK + k) * slabsz * 4;
                // transform-gradient accumulators of THIS lane for this slab: Gx[i][j] = sum xm_i * dL/dy_j and
                // Gy[j] = sum dL/dy_j; grad_rot/scale/pos are linear in them (derived once per slab, before the reduction)
#if MVP_BWD_LANESMEM
#pragma unroll
                for (int i = 0; i < 12; ++i) L_GX(i) = 0.f;
#else
                float gx[9], gsum[3];
#pragma unroll
                for (int i = 0; i < 9; ++i) gx[i] = 0.f;
                gsum[0] = gsum[1] = gsum[2] = 0.f;
#endif
                bool touched = false;
                // the step at which this lane's walk of this slab meets the ray's saturating sample (-1: never)
                const int isat_i = (rank == L_RANKSAT) ? (L_MSAT - la) : -1;
                // carry the lane's position from the chunk base (step max(cs, ms)) to its first candidate step
                float x = L_XB, y = L_YB, z = L_ZB;
                {
                    const int adv = (len > 0) ? (la - max(cs, L_MS)) : 0;
                    const int maxadv = __reduce_max_sync(0xffffffffu, adv);
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
                    if (lane == 0) std::atomic_ref<long long>(g_emul_bwd_stats[6]).fetch_add(maxadv);
#endif
                    for (int i = 0; i < maxadv; ++i) {
                        if (i < adv) { x = __fmaf_rn(rdx, p.dt, x); y = __fmaf_rn(rdy, p.dt, y); z = __fmaf_rn(rdz, p.dt, z); }
                    }
                }
                // Sample compaction: lanes enumerate their own valid steps (cheap transform + test) and push the sample
                // position into a ring; the expensive adjoint runs on full batches of 32 samples, each computed by
                // whichever lane pops it (per-ray data comes from the owner lane by shuffle; the per-slab gradient sums are
                // reduced over the warp afterwards, so it does not matter which lane accumulates a sample).
                int qhead = 0, qn = 0;
                float4 *ring = sq;
#if MVP_BWD_SMEMREC
                // The step phase (record in registers) runs until a batch is due or the interval is exhausted; the batch adjoint
                // takes what it needs of the record from shared memory; then the step phase reloads it.
                for (int i = 0;;) {
                    {
                    const Prim q = load_rec_shared(S->rec);
                    for (; i < maxlen && qn < 32; ++i) {
#else
                for (int i = 0; i <= maxlen; ++i) {
                    const bool flush = (i == maxlen);
                    if (!flush) {
#endif
                        const bool live = i < len;
                        const float xm = x - q.px, ym = y - q.py, zm = z - q.pz;
                        x = __fmaf_rn(rdx, p.dt, x); y = __fmaf_rn(rdy, p.dt, y); z = __fmaf_rn(rdz, p.dt, z);
                        const float y0 = __fmul_rn(q.sx, rowdot(q.r00, xm, q.r10, ym, q.r20, zm));
                        const float y1 = __fmul_rn(q.sy, rowdot(q.r01, xm, q.r11, ym, q.r21, zm));
                        const float y2 = __fmul_rn(q.sz, rowdot(q.r02, xm, q.r12, ym, q.r22, zm));
                        const bool valid = live && (fabsf(y0) < 1.f) && (fabsf(y1) < 1.f) && (fabsf(y2) < 1.f);   // (inside_unit here: +1.7 % instructions)
                        const unsigned vm = __ballot_sync(0xffffffffu, valid);
                        if (vm) {
                            if (valid) {
                                const int pos = (qhead + qn + __popc(vm & ((1u << lane) - 1u))) & (kRing - 1);
                                const bool issat = (i == isat_i);
                                ring[pos] = make_float4(xm, ym, zm, __int_as_float(lane | (issat ? 256 : 0)));
                            }
                            qn += __popc(vm);
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
                            if (lane == 0) std::atomic_ref<long long>(g_emul_bwd_stats[4]).fetch_add(__popc(vm));
#endif
                            __syncwarp();
                        }
                    }
#if MVP_BWD_SMEMREC
                    }
                    const bool flush = (i == maxlen);
                    if (flush && qn == 0) break;
                    {
                        const Prim q = load_rec_shared(S->rec);
#else
                    while (qn >= 32 || (flush && qn > 0)) {
#endif
#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
                        if (lane == 0) std::atomic_ref<long long>(g_emul_bwd_stats[5]).fetch_add(1);
#endif
                        const int cnt = min(qn, 32);
                        const bool act = lane < cnt;
                        const float4 rec = ring[(qhead + (act ? lane : 0)) & (kRing - 1)];
                        qhead = (qhead + cnt) & (kRing - 1);
                        qn -= cnt;
                        __syncwarp();
                        const int meta = __float_as_int(rec.w);
                        const int owner = meta & 31;
                        const bool issat = (meta & 256) != 0;
                        // per-ray data of the owner lane
                        if (!act) continue;
                        const float *pr_ = sray + owner;
                        const float oLx = pr_[0 * 32], oLy = pr_[1 * 32], oLz = pr_[2 * 32], oLw = pr_[3 * 32];
                        const float osr = pr_[4 * 32], osg = pr_[5 * 32], osb = pr_[6 * 32], osa = pr_[7 * 32], oab = pr_[8 * 32];
                        touched = true;
                        const float xm = rec.x, ym = rec.y, zm = rec.z;
                        const float rx0 = rowdot(q.r00, xm, q.r10, ym, q.r20, zm);
                        const float rx1 = rowdot(q.r01, xm, q.r11, ym, q.r21, zm);
                        const float rx2 = rowdot(q.r02, xm, q.r12, ym, q.r22, zm);
                        const float y0 = __fmul_rn(q.sx, rx0), y1 = __fmul_rn(q.sy, rx1), y2 = __fmul_rn(q.sz, rx2);
                        float gy0, gy1, gy2;   // dL/dy0 of this sample
                        if (!kWarp) {
                        // ---- forward sample (primsampler.h:44-66) keeping what the adjoint needs ----
                        const float e1 = p.fadeexp - 1.f;
                        const float pw0 = __powf(fabsf(y0), e1), pw1 = __powf(fabsf(y1), e1), pw2 = __powf(fabsf(y2), e1);
                        const float fade = __expf(-p.fadescale * (pw0 * fabsf(y0) + pw1 * fabsf(y1) + pw2 * fabsf(y2)));
                        const float fx = ((y0 + 1.f) * 0.5f) * (float)(tw - 1);
                        const float fy = ((y1 + 1.f) * 0.5f) * (float)(th - 1);
                        const float fz = ((y2 + 1.f) * 0.5f) * (float)(td - 1);
                        const int ix = __float2int_rd(fx), iy = __float2int_rd(fy), iz = __float2int_rd(fz);
                        int cx, cy, cz;
                        if (T >= 2) { cx = min(ix, T - 2); cy = min(iy, T - 2); cz = min(iz, T - 2); }
                        else { cx = max(min(ix, tw - 2), 0); cy = max(min(iy, th - 2), 0); cz = max(min(iz, td - 2), 0); }
                        const float bx0 = fx - (float)cx, bx1 = (float)(cx + 1) - fx;
                        const float by0 = fy - (float)cy, by1 = (float)(cy + 1) - fy;
                        const float bz0 = fz - (float)cz, bz1 = (float)(cz + 1) - fz;
                        const bool ex = ix > cx, ey = iy > cy, ez = iz > cz;
                        const int base = (cz * th + cy) * tw + cx;
                        const TP *pc = slab + base;
                        // One pass over the 8 corners.  dL/d(sample) = (A dL.rgb, B) with A, B known only after the sample
                        // is complete, but <T_c, dL/d(sample)> = A <T_c.rgb, dL.rgb> + B T_c.a is linear in (A, B):
                        // accumulate the index-gradient sums for both parts now and combine afterwards.
                        const float wx_[2] = {bx1, bx0}, wy_[2] = {by1, by0}, wz_[2] = {bz1, bz0};
                        float4 sv = make_float4(0.f, 0.f, 0.f, 0.f);
                        float gp[3] = {0.f, 0.f, 0.f}, ga[3] = {0.f, 0.f, 0.f};   // signed (upper - lower) corner sums per axis: rgb / alpha part
#pragma unroll
                        for (int cn = 0; cn < 8; ++cn) {
                            const int bx = cn & 1, byy = (cn >> 1) & 1, bz = (cn >> 2) & 1;
                            const float4 v = load_voxel(pc + ((bx ? sx : 0) + (byy ? sy : 0) + (bz ? sz : 0)));
                            const float w_ = (wx_[bx] * wy_[byy]) * wz_[bz];
                            sv.x = __fmaf_rn(w_, v.x, sv.x); sv.y = __fmaf_rn(w_, v.y, sv.y);
                            sv.z = __fmaf_rn(w_, v.z, sv.z); sv.w = __fmaf_rn(w_, v.w, sv.w);
                            const float pr = v.x * oLx + v.y * oLy + v.z * oLz;
                            const float wyz = wy_[byy] * wz_[bz], wxz = wx_[bx] * wz_[bz], wxy = wx_[bx] * wy_[byy];
                            // d(weight)/d(index) is +1 on the upper corner of an axis, -1 on the lower one
                            gp[0] += (bx ? pr : -pr) * wyz; ga[0] += (bx ? v.w : -v.w) * wyz;
                            gp[1] += (byy ? pr : -pr) * wxz; ga[1] += (byy ? v.w : -v.w) * wxz;
                            gp[2] += (bz ? pr : -pr) * wxy; ga[2] += (bz ? v.w : -v.w) * wxy;
                        }
                        sv.w *= fade;
                        // ---- primaccum.h:81-98 with the saturating sample known from forward ----
                        const float A = issat ? (1.f - oab) : sv.w * p.dt;             // weight of dL.rgb
                        const float dLa = issat ? 0.f : p.dt * ((sv.x - osr) * oLx + (sv.y - osg) * oLy + (sv.z - osb) * oLz + (1.f - osa) * oLw);
                        const float B = dLa * fade;                                     // dL/d(alpha0)
                        const float d0 = A * oLx, d1 = A * oLy, d2 = A * oLz;
                        // ---- primsampler.h:68-91 ----
                        const float cf = -(p.fadescale * p.fadeexp) * sv.w * dLa;
                        gy0 = cf * pw0 * (y0 > 0.f ? 1.f : -1.f);
                        gy1 = cf * pw1 * (y1 > 0.f ? 1.f : -1.f);
                        gy2 = cf * pw2 * (y2 > 0.f ? 1.f : -1.f);
                        // ---- utils.h:504-643: scatter w_c * dL_sample (zero-weight corners add 0) ----
                        float *gc = gslab + (size_t)base * 4;
#pragma unroll
                        for (int cn = 0; cn < 8; ++cn) {
                            const int o = ((cn & 1) ? sx : 0) + ((cn & 2) ? sy : 0) + ((cn & 4) ? sz : 0);
                            const float w_ = (wx_[cn & 1] * wy_[(cn >> 1) & 1]) * wz_[(cn >> 2) & 1];   // same product as above
                            red_add_v4(gc + (size_t)o * 4, w_ * d0, w_ * d1, w_ * d2, w_ * B);
                        }
                        // dL/d(index): d(weight)/d(index) is +1 on the upper corner, -1 on the lower one; on a clamped axis
                        // the reference sees the upper voxel as ITS lower corner (sign -1) and no other corner.
                        float gix = A * gp[0] + B * ga[0], giy = A * gp[1] + B * ga[1], giz = A * gp[2] + B * ga[2];
                        if (ex || ey || ez) {     // a sample exactly on a far face of the slab: see index_grad_general
                            const float3 gg = index_grad_general(pc, sx, sy, sz, bx0, bx1, by0, by1, bz0, bz1, oLx, oLy, oLz, A, B,
                                                                 (ex ? 1 : 0) | (ey ? 2 : 0) | (ez ? 4 : 0));
                            gix = gg.x; giy = gg.y; giz = gg.z;
                        }
                        gy0 += gmx * gix; gy1 += gmy * giy; gy2 += gmz * giz;
                        } else {
                        // ---- algo 1 (PrimSamplerTW<true>): payload sampled at the warp-field-displaced position ----
                        const size_t wsl = (size_t)p.WD * p.WH * p.WW * 3;
                        const float *wk = p.warp + ((size_t)(n * p.pview) * p.K + k) * wsl;
                        float *gwk = p.g_warp + ((size_t)(n * p.pview) * p.K + k) * wsl;
                        const float e1 = p.fadeexp - 1.f;
                        const float pw0 = __powf(fabsf(y0), e1), pw1 = __powf(fabsf(y1), e1), pw2 = __powf(fabsf(y2), e1);
                        const float fade = __expf(-p.fadescale * (pw0 * fabsf(y0) + pw1 * fabsf(y1) + pw2 * fabsf(y2)));
                        const CellG cw = cell_generic(y0, y1, y2, p.WD, p.WH, p.WW);
                        float u0 = 0.f, u1 = 0.f, u2 = 0.f;                    // warped position (primsampler.h:53-58)
#pragma unroll
                        for (int cn = 0; cn < 8; ++cn) {
                            if (cw.idx[cn] >= 0) {
                                const float *v = wk + (size_t)cw.idx[cn] * 3;
                                u0 = __fmaf_rn(cw.w[cn], __ldg(v), u0); u1 = __fmaf_rn(cw.w[cn], __ldg(v + 1), u1); u2 = __fmaf_rn(cw.w[cn], __ldg(v + 2), u2);
                            }
                        }
                        const CellG ct = cell_generic(u0, u1, u2, p.TD, p.TH, p.TW);
                        float4 sv = make_float4(0.f, 0.f, 0.f, 0.f);
                        float gp0 = 0.f, gp1 = 0.f, gp2 = 0.f, ga0 = 0.f, ga1 = 0.f, ga2 = 0.f;   // signed index-gradient sums (rgb / alpha part)
#pragma unroll
                        for (int cn = 0; cn < 8; ++cn) {
                            if (ct.idx[cn] >= 0) {
                                const float4 v = load_voxel(slab + ct.idx[cn]);
                                sv.x = __fmaf_rn(ct.w[cn], v.x, sv.x); sv.y = __fmaf_rn(ct.w[cn], v.y, sv.y);
                                sv.z = __fmaf_rn(ct.w[cn], v.z, sv.z); sv.w = __fmaf_rn(ct.w[cn], v.w, sv.w);
                                const float pr = v.x * oLx + v.y * oLy + v.z * oLz;
                                const float wx = (cn & 1) ? ct.x0 : ct.x1, wy = (cn & 2) ? ct.y0 : ct.y1, wz = (cn & 4) ? ct.z0 : ct.z1;
                                const float sxg = (cn & 1) ? 1.f : -1.f, syg = (cn & 2) ? 1.f : -1.f, szg = (cn & 4) ? 1.f : -1.f;
                                gp0 += sxg * pr * (wy * wz); ga0 += sxg * v.w * (wy * wz);
                                gp1 += syg * pr * (wx * wz); ga1 += syg * v.w * (wx * wz);
                                gp2 += szg * pr * (wx * wy); ga2 += szg * v.w * (wx * wy);
                            }
                        }
                        sv.w *= fade;
                        const float A = issat ? (1.f - oab) : sv.w * p.dt;
                        const float dLa = issat ? 0.f : p.dt * ((sv.x - osr) * oLx + (sv.y - osg) * oLy + (sv.z - osb) * oLz + (1.f - osa) * oLw);
                        const float B = dLa * fade;
                        const float d0 = A * oLx, d1 = A * oLy, d2 = A * oLz;
                        const float cf = -(p.fadescale * p.fadeexp) * sv.w * dLa;
                        gy0 = cf * pw0 * (y0 > 0.f ? 1.f : -1.f);
                        gy1 = cf * pw1 * (y1 > 0.f ? 1.f : -1.f);
                        gy2 = cf * pw2 * (y2 > 0.f ? 1.f : -1.f);
#pragma unroll
                        for (int cn = 0; cn < 8; ++cn)
                            if (ct.idx[cn] >= 0) red_add_v4(gslab + (size_t)ct.idx[cn] * 4, ct.w[cn] * d0, ct.w[cn] * d1, ct.w[cn] * d2, ct.w[cn] * B);
                        // dL/d(warped position)  (utils.h:591-642), then through the warp field (primsampler.h:82-88)
                        const float e0 = gmx * (A * gp0 + B * ga0), e1_ = gmy * (A * gp1 + B * ga1), e2 = gmz * (A * gp2 + B * ga2);
                        float h0 = 0.f, h1 = 0.f, h2 = 0.f;
#pragma unroll
                        for (int cn = 0; cn < 8; ++cn) {
                            if (cw.idx[cn] >= 0) {
                                const float *v = wk + (size_t)cw.idx[cn] * 3;
                                float *gv = gwk + (size_t)cw.idx[cn] * 3;
                                atomicAdd(gv, cw.w[cn] * e0); atomicAdd(gv + 1, cw.w[cn] * e1_); atomicAdd(gv + 2, cw.w[cn] * e2);
                                const float dpw = __ldg(v) * e0 + __ldg(v + 1) * e1_ + __ldg(v + 2) * e2;
                                const float wx = (cn & 1) ? cw.x0 : cw.x1, wy = (cn & 2) ? cw.y0 : cw.y1, wz = (cn & 4) ? cw.z0 : cw.z1;
                                h0 += ((cn & 1) ? dpw : -dpw) * (wy * wz);
                                h1 += ((cn & 2) ? dpw : -dpw) * (wx * wz);
                                h2 += ((cn & 4) ? dpw : -dpw) * (wx * wy);
                            }
                        }
                        gy0 += ((float)(p.WW - 1) * 0.5f) * h0; gy1 += ((float)(p.WH - 1) * 0.5f) * h1; gy2 += ((float)(p.WD - 1) * 0.5f) * h2;
                        }
                        // ---- primtransf.h:155-179, accumulated in factored form ----
#if MVP_BWD_LANESMEM
                        L_GX(0) = L_GX(0) + xm * gy0; L_GX(1) = L_GX(1) + xm * gy1; L_GX(2) = L_GX(2) + xm * gy2;
                        L_GX(3) = L_GX(3) + ym * gy0; L_GX(4) = L_GX(4) + ym * gy1; L_GX(5) = L_GX(5) + ym * gy2;
                        L_GX(6) = L_GX(6) + zm * gy0; L_GX(7) = L_GX(7) + zm * gy1; L_GX(8) = L_GX(8) + zm * gy2;
                        L_GX(9) = L_GX(9) + gy0; L_GX(10) = L_GX(10) + gy1; L_GX(11) = L_GX(11) + gy2;
#else
                        gx[0] += xm * gy0; gx[1] += xm * gy1; gx[2] += xm * gy2;
                        gx[3] += ym * gy0; gx[4] += ym * gy1; gx[5] += ym * gy2;
                        gx[6] += zm * gy0; gx[7] += zm * gy1; gx[8] += zm * gy2;
                        gsum[0] += gy0; gsum[1] += gy1; gsum[2] += gy2;
#endif
                    }
                }
                if (!__any_sync(0xffffffffu, touched)) continue;
                // grad_scale_j = sum_i R[i][j] Gx[i][j];  grad_rot[i][j] = s_j Gx[i][j];  grad_pos = -R (s * Gy)
#if MVP_BWD_SMEMREC
                const Prim q = load_rec_shared(S->rec);
#endif
#if MVP_BWD_LANESMEM
                float gx[9], gsum[3];
#pragma unroll
                for (int i = 0; i < 9; ++i) gx[i] = L_GX(i);
                gsum[0] = L_GX(9); gsum[1] = L_GX(10); gsum[2] = L_GX(11);
#endif
                float g[16];
                g[0] = q.r00 * gx[0] + q.r10 * gx[3] + q.r20 * gx[6];
                g[1] = q.r01 * gx[1] + q.r11 * gx[4] + q.r21 * gx[7];
                g[2] = q.r02 * gx[2] + q.r12 * gx[5] + q.r22 * gx[8];
                g[3] = q.sx * gx[0]; g[4] = q.sy * gx[1]; g[5] = q.sz * gx[2];
                g[6] = q.sx * gx[3]; g[7] = q.sy * gx[4]; g[8] = q.sz * gx[5];
                g[9] = q.sx * gx[6]; g[10] = q.sy * gx[7]; g[11] = q.sz * gx[8];
                {
                    const float h0 = q.sx * gsum[0], h1 = q.sy * gsum[1], h2 = q.sz * gsum[2];
                    g[12] = -(q.r00 * h0 + q.r01 * h1 + q.r02 * h2);
                    g[13] = -(q.r10 * h0 + q.r11 * h1 + q.r12 * h2);
                    g[14] = -(q.r20 * h0 + q.r21 * h1 + q.r22 * h2);
                }
                g[15] = 0.f;
                // 16-value butterfly: after the 5 stages lanes 2i and 2i+1 hold the warp total of g[i]
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const bool up = lane & 16;
                    const float send = up ? g[i] : g[i + 8];
                    const float keep = up ? g[i + 8] : g[i];
                    g[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const bool up = lane & 8;
                    const float send = up ? g[i] : g[i + 4];
                    const float keep = up ? g[i + 4] : g[i];
                    g[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                }
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const bool up = lane & 4;
                    const float send = up ? g[i] : g[i + 2];
                    const float keep = up ? g[i + 2] : g[i];
                    g[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                }
                {
                    const bool up = lane & 2;
                    const float send = up ? g[0] : g[1];
                    const float keep = up ? g[1] : g[0];
                    g[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
                }
                g[0] += __shfl_xor_sync(0xffffffffu, g[0], 1);
                const int vi = lane >> 1;
                if (!(lane & 1) && vi < 15) {
                    float *dst = vi < 3 ? (p.g_primscale + (pvK + k) * 3 + vi)
                                        : (vi < 12 ? (p.g_primrot + (pvK + k) * 9 + (vi - 3)) : (p.g_primpos + (pvK + k) * 3 + (vi - 12)));
                    atomicAdd(dst, g[0]);
                }
            }   // while (word)
        }       // for (w)
    }           // for (cs)
    return true;
}

template <int T, int CAP, bool kWarp, typename TP>
__global__ void __launch_bounds__(kWarps * 32, (CAP < kMaxHit && !kWarp) ? (MVP_BWD_MINB * 4) / kWarps : 12 / kWarps) render_backward_kernel(const Params p) {
    __shared__ BwdWarpSmem<CAP> s_w[kWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    BwdWarpSmem<CAP> *const S = &s_w[warp];
    if (CAP == kMaxHit) {
        const int cnt = *p.heavycnt;
        for (int i = blockIdx.x * kWarps + warp; i < cnt; i += gridDim.x * kWarps) {
            const int id = p.heavylist[i];
            const int tx = id % p.TXn, ty = (id / p.TXn) % p.TYn, n = id / (p.TXn * p.TYn);
            backward_tile<T, CAP, kWarp, TP>(p, n, tx, ty, lane, S);
            __syncwarp();
        }
    } else {
#if MVP_CTA_ORDER
        // 1-D grid; CTA b renders the b-th most expensive 2x2-tile block of the launch (order_ctas_kernel), or block b
        const int cid = p.use_order ? p.ctaorder[blockIdx.x] : (int)blockIdx.x;
        const int bx = cid % p.CXn, by = (cid / p.CXn) % p.CYn, n = cid / (p.CXn * p.CYn);
        const int tx = bx * kBlkTX + (warp % kBlkTX), ty = by * kBlkTY + (warp / kBlkTX);
#else
        const int tx = blockIdx.x * kBlkTX + (warp % kBlkTX), ty = blockIdx.y * kBlkTY + (warp / kBlkTX), n = blockIdx.z;
#endif
        if (tx >= p.TXn || ty >= p.TYn) return;
        if (!backward_tile<T, CAP, kWarp, TP>(p, n, tx, ty, lane, S) && lane == 0)
            p.heavylist[atomicAdd(p.heavycnt, 1)] = (n * p.TYn + ty) * p.TXn + tx;
    }
}

// Launch pair: the fast kernel over the whole tile grid, then the small persistent 512-entry kernel over the tiles the fast
// one handed over (plain stream order: it reads the heavy-tile counter the fast kernel filled).  Variadic macros because the
// kernel names contain commas.
#ifdef MVP_CPU_EMUL
#define MVP_LAUNCH_FAST(...)                                    \
    do {                                                        \
        auto kern_ = __VA_ARGS__;                               \
        MVP_LAUNCH(kern_, grid, kWarps * 32, 0, st, p);         \
    } while (0)
#define MVP_LAUNCH_HEAVY(...)                                   \
    do {                                                        \
        auto kern_ = __VA_ARGS__;                               \
        MVP_LAUNCH(kern_, dim3(kHeavyGrid), kWarps * 32, 0, st, p); \
    } while (0)
#else
#define MVP_LAUNCH_FAST(...) __VA_ARGS__<<<grid, kWarps * 32, 0, st>>>(p)
#define MVP_LAUNCH_HEAVY(...) __VA_ARGS__<<<kHeavyGrid, kWarps * 32, 0, st>>>(p)
#endif
// shared-memory carve-out preference of a fast render kernel (a per-function attribute: no allocation, no synchronisation)
#ifdef MVP_CPU_EMUL
#define MVP_CARVE(pct, ...) ((void)0)
#else
#define MVP_CARVE(pct, ...)                                                                                          \
    do {                                                                                                             \
        if ((pct) > 0) cudaFuncSetAttribute(__VA_ARGS__, cudaFuncAttributePreferredSharedMemoryCarveout, (pct));     \
    } while (0)
#endif

int check_shape(const mvp_shape &s) {
    if (s.N < 1 || s.H < 1 || s.W < 1 || s.K < 1 || s.TD < 1 || s.TH < 1 || s.TW < 1) return MVP_ERR_SHAPE;
    if (s.H >= 32768 || s.W >= 32768) return MVP_ERR_SHAPE;
    if (s.N > 65535) return MVP_ERR_SHAPE;
    if ((size_t)s.TD * s.TH * s.TW >= ((size_t)1 << 27)) return MVP_ERR_SHAPE;
    if ((size_t)s.N * ((s.H + kTileH - 1) / kTileH) * ((s.W + kTileW - 1) / kTileW) >= ((size_t)1 << 31)) return MVP_ERR_SHAPE;   // tile ids are ints
    return MVP_OK;
}

// camera: NULL or a checked mvp_camera (then raypos / raydir are not used)
int launch_accel(const mvp_shape &s, int pview, const int *order, const float *raypos, const float *raydir, const mvp_camera *camera,
                 const float *primpos, const float *primrot, const float *primscale, char *ws, const Layout &L, cudaStream_t st) {
    const int ostride = pview ? s.K : 0;      // the order belongs to the primitives: one per view, or one shared by all views
    Cam *cam = reinterpret_cast<Cam *>(ws + L.cam);
    int *bad = reinterpret_cast<int *>(ws + L.bad);
    cudaError_t e = cudaMemsetAsync(bad, 0, (size_t)s.N * sizeof(int), st);
    if (e != cudaSuccess) return (int)e;
#if MVP_LIST_REUSE
    // a new accel structure invalidates whatever lists an earlier forward saved in this workspace
    e = cudaMemsetAsync(ws + L.tilehdr, 0xff, L.listbuf - L.tilehdr, st);
    if (e != cudaSuccess) return (int)e;
#endif
    const bool want_order = MVP_CTA_ORDER && s.N <= MVP_CTA_ORDER_MAXVIEWS;
    (void)want_order;
    const bool small_launch = s.N <= MVP_CTA_ORDER_MAXVIEWS;   // latency-bound accel build: the parallel bucket kernel
    const size_t HW = (size_t)s.H * s.W;
    dim3 gfit((unsigned)((HW + kFitThreads * kFitRaysPerThread - 1) / (kFitThreads * kFitRaysPerThread)), s.N);
#ifdef MVP_CPU_EMUL
    if (camera)
        MVP_LAUNCH(cam_params_kernel, (unsigned)((s.N + 127) / 128), 128, 0, st, s.N, camera->viewpos, camera->viewrot, camera->focal,
                   camera->princpt, camera->volradius, cam, bad, reinterpret_cast<float4 *>(ws + L.raycam));
    else
        MVP_LAUNCH(fit_camera_kernel, gfit, kFitThreads, 0, st, s.H, s.W, raypos, raydir, cam, bad);
    const size_t NK = (size_t)s.N * s.K;
    MVP_LAUNCH(prim_setup_kernel, (unsigned)((NK + 127) / 128), 128, 0, st, s.N, s.K, s.H, s.W, pview, primpos, primrot, primscale, cam, bad,
               reinterpret_cast<float4 *>(ws + L.pack), reinterpret_cast<unsigned *>(ws + L.rx), reinterpret_cast<unsigned *>(ws + L.ry));
    const int TXn = (s.W + kTileW - 1) / kTileW;
    if (order) {
        const size_t nk = (size_t)(pview ? s.N : 1) * s.K;
        MVP_LAUNCH(invert_order_kernel, (unsigned)((nk + 255) / 256), 256, 0, st, nk, s.K, order, reinterpret_cast<int *>(ws + L.rankof));
    }
    MVP_LAUNCH(block_ranges_kernel, dim3(((s.K + 31) / 32 + 7) / 8, s.N), 256, 0, st, s.K, reinterpret_cast<const unsigned *>(ws + L.ry),
               order, ostride, reinterpret_cast<unsigned *>(ws + L.blky));
    if (small_launch)
        MVP_LAUNCH(row_lists_cta_kernel, dim3(L.R, s.N), kRowThreads, 0, st, s.K, L.R, L.rowcap, TXn,
                   reinterpret_cast<unsigned *>(ws + L.rx), reinterpret_cast<unsigned *>(ws + L.ry),
                   reinterpret_cast<const unsigned *>(ws + L.blky), order, ostride, reinterpret_cast<int *>(ws + L.rowcnt),
                   reinterpret_cast<RowEntry *>(ws + L.rowlist)
#if MVP_XBUCKETS
                   , L.NG, reinterpret_cast<int2 *>(ws + L.grphdr), reinterpret_cast<RowEntry *>(ws + L.grplist),
                   want_order ? reinterpret_cast<unsigned short *>(ws + L.tilecnt) : nullptr
#endif
                   );
    else
        MVP_LAUNCH(row_lists_kernel, dim3((L.R + kRowThreads / 32 - 1) / (kRowThreads / 32), s.N), kRowThreads, 0, st, s.K, L.R, L.rowcap, TXn,
                   reinterpret_cast<unsigned *>(ws + L.rx), reinterpret_cast<unsigned *>(ws + L.ry),
                   reinterpret_cast<const unsigned *>(ws + L.blky), order, ostride, reinterpret_cast<int *>(ws + L.rowcnt),
                   reinterpret_cast<RowEntry *>(ws + L.rowlist)
#if MVP_XBUCKETS
                   , L.NG, reinterpret_cast<int2 *>(ws + L.grphdr), reinterpret_cast<RowEntry *>(ws + L.grplist),
                   want_order ? reinterpret_cast<unsigned short *>(ws + L.tilecnt) : nullptr
#endif
                   );
#else
    if (camera)
        cam_params_kernel<<<(unsigned)((s.N + 127) / 128), 128, 0, st>>>(s.N, camera->viewpos, camera->viewrot, camera->focal, camera->princpt,
                                                                         camera->volradius, cam, bad, reinterpret_cast<float4 *>(ws + L.raycam));
    else
        fit_camera_kernel<<<gfit, kFitThreads, 0, st>>>(s.H, s.W, raypos, raydir, cam, bad);
    const size_t NK = (size_t)s.N * s.K;
    prim_setup_kernel<<<(unsigned)((NK + 127) / 128), 128, 0, st>>>(
        s.N, s.K, s.H, s.W, pview, primpos, primrot, primscale, cam, bad, reinterpret_cast<float4 *>(ws + L.pack),
        reinterpret_cast<unsigned *>(ws + L.rx), reinterpret_cast<unsigned *>(ws + L.ry));
    const int TXn = (s.W + kTileW - 1) / kTileW;
    if (order) {
        const size_t nk = (size_t)(pview ? s.N : 1) * s.K;
        invert_order_kernel<<<(unsigned)((nk + 255) / 256), 256, 0, st>>>(nk, s.K, order, reinterpret_cast<int *>(ws + L.rankof));
    }
    block_ranges_kernel<<<dim3(((s.K + 31) / 32 + 7) / 8, s.N), 256, 0, st>>>(s.K, reinterpret_cast<const unsigned *>(ws + L.ry), order,
                                                                               ostride, reinterpret_cast<unsigned *>(ws + L.blky));
    if (small_launch)
        row_lists_cta_kernel<<<dim3(L.R, s.N), kRowThreads, 0, st>>>(
            s.K, L.R, L.rowcap, TXn, reinterpret_cast<unsigned *>(ws + L.rx), reinterpret_cast<unsigned *>(ws + L.ry),
            reinterpret_cast<const unsigned *>(ws + L.blky), order, ostride, reinterpret_cast<int *>(ws + L.rowcnt),
            reinterpret_cast<RowEntry *>(ws + L.rowlist)
#if MVP_XBUCKETS
            , L.NG, reinterpret_cast<int2 *>(ws + L.grphdr), reinterpret_cast<RowEntry *>(ws + L.grplist),
            want_order ? reinterpret_cast<unsigned short *>(ws + L.tilecnt) : nullptr
#endif
            );
    else
        row_lists_kernel<<<dim3((L.R + kRowThreads / 32 - 1) / (kRowThreads / 32), s.N), kRowThreads, 0, st>>>(
            s.K, L.R, L.rowcap, TXn, reinterpret_cast<unsigned *>(ws + L.rx), reinterpret_cast<unsigned *>(ws + L.ry),
            reinterpret_cast<const unsigned *>(ws + L.blky), order, ostride, reinterpret_cast<int *>(ws + L.rowcnt),
            reinterpret_cast<RowEntry *>(ws + L.rowlist)
#if MVP_XBUCKETS
            , L.NG, reinterpret_cast<int2 *>(ws + L.grphdr), reinterpret_cast<RowEntry *>(ws + L.grplist),
            want_order ? reinterpret_cast<unsigned short *>(ws + L.tilecnt) : nullptr
#endif
            );
#endif
#if MVP_CTA_ORDER
    if (want_order) {
        const int TYn = L.R, CXn = (TXn + kBlkTX - 1) / kBlkTX, CYn = (TYn + kBlkTY - 1) / kBlkTY;
        const size_t ctas = (size_t)s.N * CXn * CYn;
        int *hist = reinterpret_cast<int *>(ws + L.ctahist);
        e = cudaMemsetAsync(hist, 0, 2 * kCostClasses * sizeof(int), st);
        if (e != cudaSuccess) return (int)e;
#if !MVP_XBUCKETS
        e = cudaMemsetAsync(ws + L.tilecnt, 0, (size_t)s.N * L.R * TXn * sizeof(unsigned short), st);   // no cost estimate: grid order
        if (e != cudaSuccess) return (int)e;
#endif
        for (int pass = 0; pass < 2; ++pass) {
#ifdef MVP_CPU_EMUL
            MVP_LAUNCH(order_ctas_kernel, (unsigned)((ctas + 255) / 256), 256, 0, st, pass, s.N, CXn, CYn, L.R, TXn,
                       reinterpret_cast<const unsigned short *>(ws + L.tilecnt), hist, reinterpret_cast<int *>(ws + L.ctaorder));
#else
            order_ctas_kernel<<<(unsigned)((ctas + 255) / 256), 256, 0, st>>>(pass, s.N, CXn, CYn, L.R, TXn,
                                                                              reinterpret_cast<const unsigned short *>(ws + L.tilecnt), hist,
                                                                              reinterpret_cast<int *>(ws + L.ctaorder));
#endif
        }
    }
#endif
    e = cudaGetLastError();
    return e == cudaSuccess ? MVP_OK : (int)e;
}

void fill_params(Params &p, const mvp_shape &s, float stepsize, float fadescale, float fadeexp, char *ws, const Layout &L) {
    p.N = s.N; p.H = s.H; p.W = s.W; p.K = s.K; p.TD = s.TD; p.TH = s.TH; p.TW = s.TW;
    p.dt = stepsize;
    p.fadescale = fadescale; p.fadeexp = fadeexp;
    p.pack = reinterpret_cast<const float4 *>(ws + L.pack);
    p.rx = reinterpret_cast<const unsigned *>(ws + L.rx);
    p.ry = reinterpret_cast<const unsigned *>(ws + L.ry);
    p.rowcnt = reinterpret_cast<const int *>(ws + L.rowcnt);
    p.rowlist = reinterpret_cast<const RowEntry *>(ws + L.rowlist);
    p.R = L.R; p.rowcap = L.rowcap;
    p.TXn = (s.W + kTileW - 1) / kTileW;
    p.TYn = (s.H + kTileH - 1) / kTileH;
    p.tileclk = reinterpret_cast<long long *>(ws + L.tileclk);
    p.CXn = (p.TXn + kBlkTX - 1) / kBlkTX;
    p.CYn = (p.TYn + kBlkTY - 1) / kBlkTY;
    p.ctaorder = reinterpret_cast<const int *>(ws + L.ctaorder);
    p.heavycnt = reinterpret_cast<int *>(ws + L.heavycnt);
    p.heavylist = reinterpret_cast<int *>(ws + L.heavylist);
    p.slab_bytes = (unsigned)((size_t)s.TD * s.TH * s.TW * 16);
#if MVP_XBUCKETS
    p.grphdr = reinterpret_cast<const int2 *>(ws + L.grphdr);
    p.grplist = reinterpret_cast<const RowEntry *>(ws + L.grplist);
    p.NG = L.NG;
#endif
#if MVP_LIST_REUSE
    p.tilehdr = reinterpret_cast<int2 *>(ws + L.tilehdr);
    p.listbuf = reinterpret_cast<int2 *>(ws + L.listbuf);
    p.listcur = reinterpret_cast<int *>(ws + L.listcur);
    p.rayj0 = reinterpret_cast<int *>(ws + L.rayj0);
    p.listcap = L.listcap;
    p.listlimit = L.listcap;
#endif
}

}  // namespace

extern "C" {

int mvp_abi_version(void) { return MVP_ABI_VERSION; }

int mvp_supported_flags(void) {
    return (int)(MVP_FLAG_ACCEL_VALID | MVP_FLAG_ZERO_GRADS | MVP_FLAG_SHARED_PRIMS | MVP_FLAG_TPLATE_BF16 | MVP_FLAG_TEST_TINY_LISTS);
}

#define MVP_STR2(x) #x
#define MVP_STR(x) MVP_STR2(x)
const char *mvp_build_config(void) {
    return "LIST_REUSE=" MVP_STR(MVP_LIST_REUSE)
           " LIST_MARGIN=" MVP_STR(MVP_LIST_MARGIN) " XBUCKETS=" MVP_STR(MVP_XBUCKETS) " FASTCAP=" MVP_STR(MVP_FWD_FASTCAP) "/" MVP_STR(MVP_BWD_FASTCAP) " SMEM_UNION=" MVP_STR(MVP_SMEM_UNION) " CARVEOUT=" MVP_STR(MVP_FWD_CARVEOUT) "/" MVP_STR(MVP_BWD_CARVEOUT) " FWD_RING=" MVP_STR(MVP_FWD_RING) " BWD_SMEMREC=" MVP_STR(MVP_BWD_SMEMREC) " BWD_LANESMEM=" MVP_STR(MVP_BWD_LANESMEM) " CTA_ORDER=" MVP_STR(MVP_CTA_ORDER) " CTA_ORDER_MIN=" MVP_STR(MVP_CTA_ORDER_MIN)
           " CHUNK=" MVP_STR(MVP_CHUNK) " FWD_MINB=" MVP_STR(MVP_FWD_MINB) " BWD_MINB=" MVP_STR(MVP_BWD_MINB)
           " WARPS=" MVP_STR(MVP_WARPS) " BLK_TX=" MVP_STR(MVP_BLK_TX)
#ifdef MVP_CPU_EMUL
           " CPU_EMUL"
#endif
        ;
}

const char *mvp_error_string(int code) {
    switch (code) {
        case MVP_OK: return "ok";
        case MVP_ERR_NULL: return "required pointer is NULL";
        case MVP_ERR_SHAPE: return "invalid or unsupported shape";
        case MVP_ERR_STEPSIZE: return "stepsize must be finite and > 0";
        case MVP_ERR_WORKSPACE: return "workspace too small or not 256-byte aligned";
        case MVP_ERR_ALGO: return "unsupported algo";
        case MVP_ERR_ALIGN: return "misaligned buffer (tplate/rayrgba/grad_rayrgba/grad_tplate/rayaux: 16 bytes, bf16 tplate and tminmax: 8, others: 4)";
        case MVP_ERR_STRUCT: return "args->struct_size does not match this library's argument struct (ABI mismatch)";
        case MVP_ERR_CAMERA: return "camera.volradius must be finite and > 0";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

size_t mvp_workspace_bytes(const mvp_shape *shape) {
    if (!shape || check_shape(*shape) != MVP_OK) return 0;
    return make_layout(*shape).total;
}

int mvp_build_accel(const mvp_shape *shape, uint32_t flags, const int32_t *order, const float *raypos, const float *raydir,
                    const float *primpos, const float *primrot, const float *primscale, void *workspace, size_t workspace_bytes,
                    void *stream) {
    if (!shape || !raypos || !raydir || !primpos || !primrot || !primscale || !workspace) return MVP_ERR_NULL;
    int rc = check_shape(*shape);
    if (rc != MVP_OK) return rc;
    const Layout L = make_layout(*shape);
    if (workspace_bytes < L.total || ((uintptr_t)workspace & 255)) return MVP_ERR_WORKSPACE;
    return launch_accel(*shape, (flags & MVP_FLAG_SHARED_PRIMS) ? 0 : 1, order, raypos, raydir, nullptr, primpos, primrot, primscale,
                        (char *)workspace, L, (cudaStream_t)stream);
}

// mvp_camera of an argument struct: 0 = absent, 1 = present and well-formed, < 0 = error code
static int check_camera(const mvp_camera &c) {
    const int have = (c.viewpos != nullptr) + (c.viewrot != nullptr) + (c.focal != nullptr) + (c.princpt != nullptr);
    if (have == 0) return 0;
    if (have != 4) return MVP_ERR_NULL;                                       // all four or none
    if (!(c.volradius > 0.f) || !(c.volradius < 3.0e38f)) return MVP_ERR_CAMERA;
    if (((uintptr_t)c.viewpos | (uintptr_t)c.viewrot | (uintptr_t)c.focal | (uintptr_t)c.princpt) & 3) return MVP_ERR_ALIGN;
    return 1;
}

int mvp_build_accel_camera(const mvp_shape *shape, uint32_t flags, const int32_t *order, const mvp_camera *camera, const float *primpos,
                           const float *primrot, const float *primscale, void *workspace, size_t workspace_bytes, void *stream) {
    if (!shape || !camera || !primpos || !primrot || !primscale || !workspace) return MVP_ERR_NULL;
    int rc = check_shape(*shape);
    if (rc != MVP_OK) return rc;
    rc = check_camera(*camera);
    if (rc <= 0) return rc == 0 ? MVP_ERR_NULL : rc;
    const Layout L = make_layout(*shape);
    if (workspace_bytes < L.total || ((uintptr_t)workspace & 255)) return MVP_ERR_WORKSPACE;
    return launch_accel(*shape, (flags & MVP_FLAG_SHARED_PRIMS) ? 0 : 1, order, nullptr, nullptr, camera, primpos, primrot, primscale,
                        (char *)workspace, L, (cudaStream_t)stream);
}

int mvp_debug_saved_tiles(const mvp_shape *shape, const void *host_workspace_copy, int *saved, int *not_saved) {
    if (!shape || !host_workspace_copy || !saved || !not_saved || check_shape(*shape) != MVP_OK) return MVP_ERR_NULL;
    *saved = *not_saved = 0;
#if MVP_LIST_REUSE
    const Layout L = make_layout(*shape);
    const size_t tiles = (size_t)shape->N * ((shape->H + kTileH - 1) / kTileH) * ((shape->W + kTileW - 1) / kTileW);
    const int2 *hdr = reinterpret_cast<const int2 *>((const char *)host_workspace_copy + L.tilehdr);
    for (size_t i = 0; i < tiles; ++i) {
        if (hdr[i].y > 0) ++*saved;
        else if (hdr[i].y < 0) ++*not_saved;
    }
#endif
    return MVP_OK;
}

size_t mvp_debug_tileclk_offset(const mvp_shape *shape) {
    if (!shape || check_shape(*shape) != MVP_OK) return 0;
    return make_layout(*shape).tileclk;
}

int mvp_forward_launch_count(uint32_t flags) { return (flags & MVP_FLAG_ACCEL_VALID) ? 2 : 6; }   // + 2 ordering kernels for small launches
int mvp_backward_launch_count(uint32_t flags) { return (flags & MVP_FLAG_ACCEL_VALID) ? 2 : 6; }

static inline bool misaligned(const void *p, uintptr_t a) { return p && ((uintptr_t)p & (a - 1)); }

int mvp_raymarch_forward(const mvp_forward_args *a, void *stream) {
    if (!a) return MVP_ERR_NULL;
    if (a->struct_size != sizeof(mvp_forward_args)) return MVP_ERR_STRUCT;
    const int camrc = check_camera(a->camera);
    if (camrc < 0) return camrc;
    const mvp_camera *const camera = camrc ? &a->camera : nullptr;      // rays generated in the kernels: the ray tensors are not read
    if ((!camera && (!a->raypos || !a->raydir || !a->tminmax)) || !a->primpos || !a->primrot || !a->primscale || !a->tplate || !a->workspace)
        return MVP_ERR_NULL;
    if ((a->rayrgb_nchw == nullptr) != (a->rayalpha_nchw == nullptr)) return MVP_ERR_NULL;
    if (!a->rayrgba && !a->rayrgb_nchw) return MVP_ERR_NULL;          // at least one form of the output
    if ((a->raysat == nullptr) != (a->rayaux == nullptr)) return MVP_ERR_NULL;
    int rc = check_shape(a->shape);
    if (rc != MVP_OK) return rc;
    if (a->algo != 0 && a->algo != 1) return MVP_ERR_ALGO;
    if (a->algo == 1 && (!a->warp || a->WD < 1 || a->WH < 1 || a->WW < 1)) return a->warp ? MVP_ERR_SHAPE : MVP_ERR_NULL;
    if (!(a->stepsize > 0.f) || !(a->stepsize < 3.0e38f)) return MVP_ERR_STEPSIZE;
    const Layout L = make_layout(a->shape);
    if (a->workspace_bytes < L.total || ((uintptr_t)a->workspace & 255)) return MVP_ERR_WORKSPACE;
    const bool bf16 = (a->flags & MVP_FLAG_TPLATE_BF16) != 0;
    // vector accesses: float4 (tplate, rayrgba), int4 (rayaux), float2 (tminmax); everything else is read as scalars.  A bf16 tplate
    // is read as 8-byte voxels.
    if (misaligned(a->tplate, bf16 ? 8 : 16) || misaligned(a->rayrgba, 16) || misaligned(a->rayaux, 16) || misaligned(a->tminmax, 8) ||
        misaligned(a->raypos, 4) || misaligned(a->raydir, 4) || misaligned(a->primpos, 4) || misaligned(a->primrot, 4) ||
        misaligned(a->primscale, 4) || misaligned(a->raysat, 4) || misaligned(a->warp, 4) || misaligned(a->rayrgb_nchw, 4) ||
        misaligned(a->rayalpha_nchw, 4) || misaligned(a->order, 4) || misaligned(a->clear_grad_primpos, 16) ||
        misaligned(a->clear_grad_primrot, 16) || misaligned(a->clear_grad_primscale, 16) || misaligned(a->clear_grad_tplate, 16) ||
        misaligned(a->clear_grad_warp, 16))
        return MVP_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)a->workspace;
    const int pview = (a->flags & MVP_FLAG_SHARED_PRIMS) ? 0 : 1;
    if (!(a->flags & MVP_FLAG_ACCEL_VALID)) {
        rc = launch_accel(a->shape, pview, a->order, a->raypos, a->raydir, camera, a->primpos, a->primrot, a->primscale, ws, L, st);
        if (rc != MVP_OK) return rc;
    }
    Params p{};
    fill_params(p, a->shape, a->stepsize, a->fadescale, a->fadeexp, ws, L);
    p.pview = pview;
    p.raycam = camera ? reinterpret_cast<const float4 *>(ws + L.raycam) : nullptr;
    p.order = a->order; p.rankof = a->order ? reinterpret_cast<const int *>(ws + L.rankof) : nullptr;
    p.rgb_nchw = a->rayrgb_nchw; p.alpha_nchw = a->rayalpha_nchw;
#if MVP_LIST_REUSE
    if (a->flags & MVP_FLAG_TEST_TINY_LISTS) p.listlimit = p.listcap < 16 ? p.listcap : 16;
#endif
    p.use_order = a->shape.N <= MVP_CTA_ORDER_MAXVIEWS;
    p.raypos = a->raypos; p.raydir = a->raydir; p.tminmax = a->tminmax; p.tplate = a->tplate;
    if (bf16) p.slab_bytes /= 2;
    p.rayrgba = a->rayrgba; p.raysat = a->raysat; p.rayaux = reinterpret_cast<int4 *>(a->rayaux);
    p.warp = a->warp; p.WD = a->WD; p.WH = a->WH; p.WW = a->WW;
#if MVP_CTA_ORDER
    dim3 grid((unsigned)((size_t)p.CXn * p.CYn * a->shape.N));
#else
    dim3 grid(p.CXn, p.CYn, a->shape.N);
    if (grid.y > 65535) return MVP_ERR_SHAPE;
#endif
    {
        cudaError_t e0 = cudaMemsetAsync(p.heavycnt, 0, sizeof(int), st);
        if (e0 != cudaSuccess) return (int)e0;
    }
    if (a->raysat) {
        // gradient buffers to clear for the coming backward: in the fast render kernel (one slice per warp), see clear_grad_slices
        const size_t nk = (size_t)(pview ? a->shape.N : 1) * a->shape.K;
        float *const bufs[kClearBufs] = {a->clear_grad_primpos, a->clear_grad_primrot, a->clear_grad_primscale, a->clear_grad_tplate,
                                         a->algo == 1 ? a->clear_grad_warp : nullptr};
        const size_t floats[kClearBufs] = {nk * 3, nk * 9, nk * 3, nk * a->shape.TD * a->shape.TH * a->shape.TW * 4,
                                           a->algo == 1 ? nk * a->WD * a->WH * a->WW * 3 : 0};
        for (int b = 0; b < kClearBufs; ++b) {
            if (!bufs[b]) continue;
#if MVP_CTA_ORDER
            const size_t G = (size_t)grid.x * kWarps, n4 = floats[b] / 4;
            p.clr[b] = bufs[b]; p.clrn[b] = floats[b]; p.clrper[b] = (n4 + G - 1) / G;
#else
            cudaError_t z = cudaMemsetAsync(bufs[b], 0, floats[b] * sizeof(float), st);
            if (z != cudaSuccess) return (int)z;
#endif
        }
    }
#if MVP_LIST_REUSE
    if (a->raysat) {
        cudaError_t e0 = cudaMemsetAsync(p.listcur, 0, (size_t)a->shape.N * sizeof(int), st);
        if (e0 != cudaSuccess) return (int)e0;
    }
#endif
    const int cubic = (a->shape.TD == a->shape.TH && a->shape.TH == a->shape.TW) ? a->shape.TD : 0;
#define MVP_LAUNCH_FWD(TT, WW_, TP_)                                                                         \
    do {                                                                                                     \
        if (a->raysat) {                                                                                     \
            MVP_CARVE(MVP_FWD_CARVEOUT, render_forward_kernel<TT, true, kFastCapF, WW_, TP_>);               \
            MVP_LAUNCH_FAST(render_forward_kernel<TT, true, kFastCapF, WW_, TP_>);                           \
            MVP_LAUNCH_HEAVY(render_forward_kernel<TT, true, kMaxHit, WW_, TP_>);                            \
        } else {                                                                                             \
            MVP_CARVE(MVP_FWD_CARVEOUT, render_forward_kernel<TT, false, kFastCapF, WW_, TP_>);              \
            MVP_LAUNCH_FAST(render_forward_kernel<TT, false, kFastCapF, WW_, TP_>);                          \
            MVP_LAUNCH_HEAVY(render_forward_kernel<TT, false, kMaxHit, WW_, TP_>);                           \
        }                                                                                                    \
    } while (0)
#define MVP_LAUNCH_FWD_T(TP_)                                                                                \
    do {                                                                                                     \
        if (a->algo == 1) MVP_LAUNCH_FWD(0, true, TP_);                                                      \
        else if (cubic == 8) MVP_LAUNCH_FWD(8, false, TP_);                                                  \
        else if (cubic == 16) MVP_LAUNCH_FWD(16, false, TP_);                                                \
        else MVP_LAUNCH_FWD(0, false, TP_);                                                                  \
    } while (0)
    if (bf16) MVP_LAUNCH_FWD_T(uint2);
    else MVP_LAUNCH_FWD_T(float4);
#undef MVP_LAUNCH_FWD_T
#undef MVP_LAUNCH_FWD
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? MVP_OK : (int)e;
}

int mvp_raymarch_backward(const mvp_backward_args *a, void *stream) {
    if (!a) return MVP_ERR_NULL;
    if (a->struct_size != sizeof(mvp_backward_args)) return MVP_ERR_STRUCT;
    const int camrc = check_camera(a->camera);
    if (camrc < 0) return camrc;
    const mvp_camera *const camera = camrc ? &a->camera : nullptr;
    if ((!camera && (!a->raypos || !a->raydir || !a->tminmax)) || !a->primpos || !a->primrot || !a->primscale || !a->tplate ||
        !a->raysat || !a->rayaux || !a->grad_primpos || !a->grad_primrot || !a->grad_primscale ||
        !a->grad_tplate || !a->workspace)
        return MVP_ERR_NULL;
    // the image gradient: channels-last [N,H,W,4], or as image planes (both of them, and then not the other form)
    if ((a->grad_rayrgb_nchw == nullptr) != (a->grad_rayalpha_nchw == nullptr)) return MVP_ERR_NULL;
    if ((a->grad_rayrgba == nullptr) == (a->grad_rayrgb_nchw == nullptr)) return MVP_ERR_NULL;
    int rc = check_shape(a->shape);
    if (rc != MVP_OK) return rc;
    if (a->algo != 0 && a->algo != 1) return MVP_ERR_ALGO;
    if (a->algo == 1 && (!a->warp || !a->grad_warp || a->WD < 1 || a->WH < 1 || a->WW < 1)) return (a->warp && a->grad_warp) ? MVP_ERR_SHAPE : MVP_ERR_NULL;
    if (!(a->stepsize > 0.f) || !(a->stepsize < 3.0e38f)) return MVP_ERR_STEPSIZE;
    const Layout L = make_layout(a->shape);
    if (a->workspace_bytes < L.total || ((uintptr_t)a->workspace & 255)) return MVP_ERR_WORKSPACE;
    const bool bf16 = (a->flags & MVP_FLAG_TPLATE_BF16) != 0;   // tplate only: the gradient stays fp32
    if (misaligned(a->tplate, bf16 ? 8 : 16) || misaligned(a->grad_tplate, 16) || misaligned(a->grad_rayrgba, 16) || misaligned(a->rayaux, 16) ||
        misaligned(a->tminmax, 8) || misaligned(a->raypos, 4) || misaligned(a->raydir, 4) || misaligned(a->primpos, 4) ||
        misaligned(a->primrot, 4) || misaligned(a->primscale, 4) || misaligned(a->raysat, 4) || misaligned(a->grad_primpos, 4) ||
        misaligned(a->grad_primrot, 4) || misaligned(a->grad_primscale, 4) || misaligned(a->warp, 4) || misaligned(a->grad_warp, 4) ||
        misaligned(a->grad_rayrgb_nchw, 4) || misaligned(a->grad_rayalpha_nchw, 4) || misaligned(a->order, 4))
        return MVP_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)a->workspace;
    const int pview = (a->flags & MVP_FLAG_SHARED_PRIMS) ? 0 : 1;
    if (!(a->flags & MVP_FLAG_ACCEL_VALID)) {
        rc = launch_accel(a->shape, pview, a->order, a->raypos, a->raydir, camera, a->primpos, a->primrot, a->primscale, ws, L, st);
        if (rc != MVP_OK) return rc;
    }
    if (a->flags & MVP_FLAG_ZERO_GRADS) {
        const size_t nk = (size_t)(pview ? a->shape.N : 1) * a->shape.K;
        cudaError_t z = cudaMemsetAsync(a->grad_primpos, 0, nk * 3 * sizeof(float), st);
        if (z == cudaSuccess) z = cudaMemsetAsync(a->grad_primrot, 0, nk * 9 * sizeof(float), st);
        if (z == cudaSuccess) z = cudaMemsetAsync(a->grad_primscale, 0, nk * 3 * sizeof(float), st);
        if (z == cudaSuccess) z = cudaMemsetAsync(a->grad_tplate, 0, nk * a->shape.TD * a->shape.TH * a->shape.TW * 4 * sizeof(float), st);
        if (z == cudaSuccess && a->algo == 1) z = cudaMemsetAsync(a->grad_warp, 0, nk * a->WD * a->WH * a->WW * 3 * sizeof(float), st);
        if (z != cudaSuccess) return (int)z;
    }
    Params p{};
    fill_params(p, a->shape, a->stepsize, a->fadescale, a->fadeexp, ws, L);
    p.pview = pview;
    p.raycam = camera ? reinterpret_cast<const float4 *>(ws + L.raycam) : nullptr;
    p.raypos = a->raypos; p.raydir = a->raydir; p.tminmax = a->tminmax; p.tplate = a->tplate;
    if (bf16) p.slab_bytes /= 2;
    p.use_order = a->shape.N <= MVP_CTA_ORDER_MAXVIEWS;
    p.order = a->order; p.rankof = a->order ? reinterpret_cast<const int *>(ws + L.rankof) : nullptr;
    p.g_rgb_nchw = a->grad_rayrgb_nchw; p.g_alpha_nchw = a->grad_rayalpha_nchw;
    p.grad_rayrgba = a->grad_rayrgba; p.raysat_in = a->raysat; p.rayaux_in = reinterpret_cast<const int4 *>(a->rayaux);
    p.g_primpos = a->grad_primpos; p.g_primrot = a->grad_primrot; p.g_primscale = a->grad_primscale; p.g_tplate = a->grad_tplate;
    p.warp = a->warp; p.g_warp = a->grad_warp; p.WD = a->WD; p.WH = a->WH; p.WW = a->WW;
#if MVP_CTA_ORDER
    dim3 grid((unsigned)((size_t)p.CXn * p.CYn * a->shape.N));
#else
    dim3 grid(p.CXn, p.CYn, a->shape.N);
    if (grid.y > 65535) return MVP_ERR_SHAPE;
#endif
    {
        cudaError_t e0 = cudaMemsetAsync(p.heavycnt, 0, sizeof(int), st);
        if (e0 != cudaSuccess) return (int)e0;
    }
    const int cubic = (a->shape.TD == a->shape.TH && a->shape.TH == a->shape.TW) ? a->shape.TD : 0;
#define MVP_LAUNCH_BWD(TT, WW_, TP_)                                                             \
    do {                                                                                         \
        MVP_CARVE(MVP_BWD_CARVEOUT, render_backward_kernel<TT, kFastCapB, WW_, TP_>);            \
        MVP_LAUNCH_FAST(render_backward_kernel<TT, kFastCapB, WW_, TP_>);                        \
        MVP_LAUNCH_HEAVY(render_backward_kernel<TT, kMaxHit, WW_, TP_>);                         \
    } while (0)
#define MVP_LAUNCH_BWD_T(TP_)                                                                    \
    do {                                                                                         \
        if (a->algo == 1) MVP_LAUNCH_BWD(0, true, TP_);                                          \
        else if (cubic == 8) MVP_LAUNCH_BWD(8, false, TP_);                                      \
        else if (cubic == 16) MVP_LAUNCH_BWD(16, false, TP_);                                    \
        else MVP_LAUNCH_BWD(0, false, TP_);                                                      \
    } while (0)
    if (bf16) MVP_LAUNCH_BWD_T(uint2);
    else MVP_LAUNCH_BWD_T(float4);
#undef MVP_LAUNCH_BWD_T
#undef MVP_LAUNCH_BWD
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? MVP_OK : (int)e;
}

#if defined(MVP_CPU_EMUL) && defined(MVP_EMUL_STATS)
void mvp_emul_fwd_stats(long long *out) {
    for (int i = 0; i < 8; ++i) { out[i] = g_emul_fwd_stats[i]; g_emul_fwd_stats[i] = 0; }
}
void mvp_emul_fwd_stats2(long long *out) {
    for (int i = 0; i < 8; ++i) { out[i] = g_emul_fwd_stats2[i]; g_emul_fwd_stats2[i] = 0; }
}
void mvp_emul_bwd_stats(long long *out) {
    for (int i = 0; i < 8; ++i) { out[i] = g_emul_bwd_stats[i]; g_emul_bwd_stats[i] = 0; }
}
long long mvp_emul_list_chunks(void) { const long long v = g_emul_list_chunks; g_emul_list_chunks = 0; return v; }
#endif
#if defined(MVP_CPU_EMUL) && MVP_LIST_REUSE
void mvp_emul_saved_list_tiles(int *loaded, int *rebuilt) {
    *loaded = g_emul_saved_list_tiles[0]; *rebuilt = g_emul_saved_list_tiles[1];
    g_emul_saved_list_tiles[0] = g_emul_saved_list_tiles[1] = 0;
}
#endif

}  // extern "C"
