/*
 * mvpraymarch_b200 -- C-ABI of the B200-native (sm_100a) MVP raymarcher.
 *
 * This is the drop-in boundary for ava-256's hot path: every entry point below replaces one function of
 * the reference's pybind11 module `mvpraymarchlib` (reference paths relative to /root/reference):
 *
 *   mvp_raymarch_forward   <- raymarch_forward   extensions/mvpraymarch/mvpraymarch.cpp:180-280
 *                             (+ compute_aabb    extensions/mvpraymarch/mvpraymarch.cpp:146-178, which the
 *                              reference's Python calls right before it, mvpraymarch.py:81-82: building the
 *                              acceleration structure is part of the forward call here)
 *   mvp_raymarch_backward  <- raymarch_backward  extensions/mvpraymarch/mvpraymarch.cpp:282-396
 *   mvp_build_accel        <- compute_aabb       extensions/mvpraymarch/mvpraymarch.cpp:146-178
 *                             (stand-alone form, for callers that want to build once and march many times)
 *   mvp_workspace_bytes    <- the tensors build_accel allocates, extensions/mvpraymarch/mvpraymarch.py:21-84
 *   mvp_compute_raydirs    <- compute_raydirs_forward  extensions/utils/utils.cpp:46-82 (pybind module `utilslib`;
 *                             the step right before the raymarcher, SURVEY.md section 8f row 1)
 *   mvp_camera (struct)    <- the same call fused away: given the camera parameters compute_raydirs takes
 *                             (models/autoencoder.py:240), the render kernels generate each tile's rays in their prologue
 *                             (extensions/utils/utils_kernel.cu:32-46) and raypos / raydir / tminmax never exist in HBM
 *
 * and two entry points that replace eager PyTorch chains of the callers either side of the path (no native reference
 * counterpart; SURVEY.md section 8f rows 2 and 4):
 *
 *   mvp_composite_*        <- models/raymarchers/mvpraymarcher.py:50-51 (NHWC -> NCHW rgb / alpha split),
 *                             models/colorcals/colorcal.py:26-29 (w * rgb + b), models/autoencoder.py:262-270 (matting)
 *   mvp_assemble_payload_* <- models/decoders/rgb.py:128-143, models/decoders/geometry.py:180-185 (image -> slab
 *                             re-layout), models/decoders/assembler.py:261 (relu(rgb * 25 + 100), relu(alpha), cat)
 *
 * Conventions (same ownership model as the reference: the caller owns every buffer, outputs are written in
 * place; unlike the reference nothing is allocated inside and everything runs on the caller's stream):
 *   - all pointers are DEVICE pointers to contiguous fp32 (or int32) arrays; no torch types; the one exception is a bf16
 *     tplate under MVP_FLAG_TPLATE_BF16;
 *   - `stream` is a cudaStream_t passed as void*;
 *   - return value: 0 = ok, < 0 = invalid argument (MVP_ERR_*), > 0 = a cudaError_t from the launch;
 *   - thread-safe and re-entrant: no global state.
 *
 * Tensor layouts (SURVEY.md terminology table):
 *   raypos, raydir [N,H,W,3]   tminmax [N,H,W,2]
 *   primpos [N,K,3]  primrot [N,K,3,3] (row-major)  primscale [N,K,3] (inverse half-extents)
 *   tplate  [N,K,TD,TH,TW,4] channels-last RGBA, fp32 or (MVP_FLAG_TPLATE_BF16) bf16; grad_tplate is fp32 either way
 *   warp [N,K,WD,WH,WW,3] channels-last (algo 1)
 *   rayrgba [N,H,W,4]  raysat [N,H,W,3]  rayaux [N,H,W,4] (int32, opaque; written by forward, read by backward)
 */
#ifndef MVPRAYMARCH_B200_H_
#define MVPRAYMARCH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVP_ABI_VERSION 8

#define MVP_OK 0
#define MVP_ERR_NULL (-1)      /* a required pointer is NULL */
#define MVP_ERR_SHAPE (-2)     /* non-positive or unsupported dimension (H, W < 32768; K >= 1) */
#define MVP_ERR_STEPSIZE (-3)  /* stepsize must be finite and > 0 */
#define MVP_ERR_WORKSPACE (-4) /* workspace too small or misaligned (256 B) */
#define MVP_ERR_ALGO (-5)      /* algo must be 0 (no warp field) or 1 (warp field, primsampler.h:53-58) */
#define MVP_ERR_ALIGN (-6)     /* a vector-accessed buffer is misaligned: tplate, rayrgba, grad_rayrgba, grad_tplate, rayaux
                                * need 16 bytes, a bf16 tplate (MVP_FLAG_TPLATE_BF16) and tminmax 8, everything else 4 */
#define MVP_ERR_STRUCT (-7)    /* args->struct_size != sizeof(the struct this library was built with) */
#define MVP_ERR_CAMERA (-8)    /* camera.volradius must be finite and > 0 */

typedef struct mvp_shape {
    int32_t N, H, W, K, TD, TH, TW;
} mvp_shape;

/* flags */
#define MVP_FLAG_ACCEL_VALID 1u /* workspace already holds the accel structure of these primitives+rays */
#define MVP_FLAG_ZERO_GRADS 2u  /* backward only: the library zero-fills the gradient buffers on `stream` before it
                                 * accumulates into them (replaces the caller's zeros_like of mvpraymarch.py:240-246) */
#define MVP_FLAG_SHARED_PRIMS 4u /* primpos/primrot/primscale/tplate/warp (and their gradients) have a batch dimension of
                                 * ONE that all N views share: [1,K,...] instead of [N,K,...] (SURVEY.md section 8e
                                 * "optional fast path"); gradients of all views accumulate into the one set.  Must be the
                                 * same in mvp_build_accel / forward / backward calls that share a workspace. */
#define MVP_FLAG_TPLATE_BF16 8u  /* forward and backward: tplate holds bfloat16 [N,K,TD,TH,TW,4] ([1,K,...] with
                                 * MVP_FLAG_SHARED_PRIMS), 8-byte aligned, instead of fp32.  Each voxel is converted to fp32 on
                                 * load (exact), so the result is the fp32 call's on the same values.  grad_tplate and
                                 * clear_grad_tplate stay fp32.  Must be the same in a forward and the backward that shares its
                                 * workspace.  Check mvp_supported_flags() before setting it. */
#define MVP_FLAG_TEST_TINY_LISTS 0x100u /* test hook: forward keeps at most 16 saved tile-list entries per view, so almost
                                 * every tile takes the backward's rebuild path */

/* The pinhole cameras of the N views, exactly the arguments of the reference's compute_raydirs (extensions/utils/utils.py:21-51,
 * kernel utils_kernel.cu:12-52) on the integer pixel grid (its `pixelcoords` = (W, H) tuple form): ray (n, h, w) starts at
 * viewpos[n] / volradius and points along normalize(viewrot[n]^T ((w - princpt.x) / focal.x, (h - princpt.y) / focal.y, 1)).
 * A call that gets a camera (viewpos != NULL) generates the rays inside the kernels -- bit-identical to what
 * mvp_compute_raydirs writes -- and ignores raypos / raydir / tminmax, which may then be NULL: 32 bytes per ray that are neither
 * written by a ray-generation pass nor read by forward and backward, and no camera fit over the ray field in the accel build.
 * All four pointers or none; volradius finite and > 0.  Must be the same in every call that shares a workspace. */
typedef struct mvp_camera {
    const float *viewpos;    /* [N,3]   camera centres (same unit as volradius) */
    const float *viewrot;    /* [N,3,3] row-major; rows = camera x, y, z axes in world coordinates */
    const float *focal;      /* [N,2]   focal lengths in pixels (x, y) */
    const float *princpt;    /* [N,2]   principal point in pixels (x, y) */
    float volradius;         /* world units of the unit cube's half edge (models/autoencoder.py: self.volradius) */
    uint32_t reserved;       /* 0 */
} mvp_camera;

typedef struct mvp_forward_args {
    uint32_t struct_size;    /* = sizeof(mvp_forward_args); a truncated or stale caller-side struct is rejected */
    mvp_shape shape;
    float stepsize, fadescale, fadeexp;
    uint32_t flags;
    const float *raypos, *raydir, *tminmax;   /* may be NULL when `camera` is given */
    const float *primpos, *primrot, *primscale;
    const float *tplate;
    float *rayrgba;          /* out; may be NULL when rayrgb_nchw / rayalpha_nchw are given */
    float *raysat;           /* out, NULL when no gradient will be taken (mvpraymarch.py:147-152) */
    int32_t *rayaux;         /* out, NULL iff raysat is NULL */
    void *workspace;         /* >= mvp_workspace_bytes(shape), 256-byte aligned */
    size_t workspace_bytes;
    /* algo 1 only (reference: PrimSamplerTW<true>): warp field [N,K,WD,WH,WW,3] channels-last, sampled at the slab
     * coordinate; the payload is then sampled at the warped position (zero outside the slab).  algo 0 ignores these. */
    const float *warp;
    int32_t WD, WH, WW;
    int32_t algo;            /* 0 or 1 (mvpraymarch.py:303) */
    /* Optional image-plane outputs, written by the render kernel's epilogue (both or neither): rayrgb [N,3,H,W] and
     * rayalpha [N,1,H,W] -- what models/raymarchers/mvpraymarcher.py:50-51 makes of rayrgba with a permute and two
     * .contiguous() copies (SURVEY.md section 8f row 2). */
    float *rayrgb_nchw;
    float *rayalpha_nchw;
    /* Optional marching order [N,K] int32 ([1,K] with MVP_FLAG_SHARED_PRIMS): order[n][j] = index of the slab marched j-th.
     * NULL = the reference's fixed order (utils.h:740-742).  This is the `sortedobjid` of the reference's usebvh=True branch
     * (mvpraymarch.py:46-55; codes from mvp_compute_morton) applied as an indirection instead of a gather of the primitive
     * tensors.  Must be a permutation of 0..K-1 and the same in every call that shares the workspace. */
    const int32_t *order;
    /* Optional (each may be NULL): the gradient buffers of the mvp_raymarch_backward call that will follow, shapes as in
     * mvp_backward_args.  A gradient-mode forward (raysat != NULL) zero-fills them from inside its render kernel -- every warp
     * clears one slice with streaming stores before it renders its tile; the kernel is issue bound and the DRAM write path idle,
     * so the 134 MB per view cost nothing measurable, where a memset pass (MVP_FLAG_ZERO_GRADS in the backward, or the caller's
     * zeros_like of mvpraymarch.py:265-268) costs 1.4 ms per 80 views.  16-byte aligned; ignored when raysat is NULL;
     * clear_grad_warp is used for algo 1 only. */
    float *clear_grad_primpos, *clear_grad_primrot, *clear_grad_primscale, *clear_grad_tplate, *clear_grad_warp;
    mvp_camera camera;       /* optional (camera.viewpos != NULL): rays generated in the kernels, see mvp_camera */
} mvp_forward_args;

typedef struct mvp_backward_args {
    uint32_t struct_size;    /* = sizeof(mvp_backward_args) */
    mvp_shape shape;
    float stepsize, fadescale, fadeexp;
    uint32_t flags;          /* MVP_FLAG_ACCEL_VALID if `workspace` is the one the forward call filled: besides the accel
                              * structure it then holds each tile's slab list and each ray's first step as the forward (called
                              * with raysat != NULL) saved them, and the backward loads them instead of rebuilding; without the
                              * flag, or for tiles that did not fit, everything is rebuilt from the inputs */
    const float *raypos, *raydir, *tminmax;
    const float *primpos, *primrot, *primscale;
    const float *tplate;
    const float *grad_rayrgba; /* [N,H,W,4]; NULL when the gradient comes as image planes (grad_rayrgb_nchw / grad_rayalpha_nchw) */
    const float *raysat;       /* from forward */
    const int32_t *rayaux;     /* from forward */
    float *grad_primpos, *grad_primrot, *grad_primscale; /* out, accumulated into: caller zero-fills (or MVP_FLAG_ZERO_GRADS) */
    float *grad_tplate;        /* out, accumulated into: caller zero-fills (or MVP_FLAG_ZERO_GRADS) */
    void *workspace;
    size_t workspace_bytes;
    const float *warp;         /* algo 1 only */
    float *grad_warp;          /* algo 1 only; out, accumulated into: caller zero-fills */
    int32_t WD, WH, WW;
    int32_t algo;
    /* The incoming gradient as image planes [N,3,H,W] + [N,1,H,W] (both, with grad_rayrgba == NULL), read by the kernel's
     * prologue: the adjoint of the fused epilogue above; replaces the contiguous() copy of mvpraymarch.py:264. */
    const float *grad_rayrgb_nchw;
    const float *grad_rayalpha_nchw;
    const int32_t *order;      /* as in the forward call */
    mvp_camera camera;         /* as in the forward call */
} mvp_backward_args;

int mvp_abi_version(void);
/* The MVP_FLAG_* bits this library understands (a caller checks a newer flag here before it sets it). */
int mvp_supported_flags(void);
/* Build-time knobs of the kernels in this library, e.g. "FWD_OPAQUE=2 LIST_REUSE=1 ..." (for bench / bug reports). */
const char *mvp_build_config(void);
const char *mvp_error_string(int code);

/* Bytes of scratch the accel structure + per-call state need for this shape (0 for an invalid shape). */
size_t mvp_workspace_bytes(const mvp_shape *shape);

/* Build the acceleration structure (camera fit, primitive records, screen rectangles, tile-row lists). */
int mvp_build_accel(const mvp_shape *shape, uint32_t flags, const int32_t *order, const float *raypos, const float *raydir,
                    const float *primpos, const float *primrot, const float *primscale,
                    void *workspace, size_t workspace_bytes, void *stream);
/* The same from the camera parameters instead of the ray field (see mvp_camera): no pass over the rays at all. */
int mvp_build_accel_camera(const mvp_shape *shape, uint32_t flags, const int32_t *order, const mvp_camera *camera,
                           const float *primpos, const float *primrot, const float *primscale,
                           void *workspace, size_t workspace_bytes, void *stream);

/* 30-bit Morton codes of slab centres that the caller has normalised to the unit cube (mvpraymarch.py:46-50):
 * compute_morton of the reference (extensions/mvpraymarch/mvpraymarch.cpp:106-121, bvh.cu:20-57).
 * centre [N,K,3] -> code [N,K] int32.  Sorting a view's codes gives the `order` the raymarch calls take. */
int mvp_compute_morton(int32_t N, int32_t K, const float *centre, int32_t *code, void *stream);

int mvp_raymarch_forward(const mvp_forward_args *args, void *stream);
int mvp_raymarch_backward(const mvp_backward_args *args, void *stream);

/* Pinhole ray generation + unit-cube clip (reference: extensions/utils/utils_kernel.cu:12-52).
 * viewpos [N,3], viewrot [N,3,3], focal [N,2], princpt [N,2], pixelcoords [N,H,W,2] or NULL (integer grid);
 * outputs raypos, raydir [N,H,W,3], tminmax [N,H,W,2]. */
int mvp_compute_raydirs(int32_t N, int32_t H, int32_t W, const float *viewpos, const float *viewrot, const float *focal,
                        const float *princpt, const float *pixelcoords, float volradius, float *raypos, float *raydir,
                        float *tminmax, void *stream);

/* Image epilogue (SURVEY.md section 8f row 2).  rayrgba [N,H,W,4] (16-byte aligned) ->
 *   irgbrec  [N,3,H,W] = (ccw[n,c] * rgb + ccb[n,c]) + (1 - alpha) * bg[n,c,h,w]      (each op rounded once, like eager torch)
 *   rayalpha [N,1,H,W] = alpha                                                        (optional)
 * ccw, ccb [N,3]: per-view colour calibration, both NULL for none; bg [N,3,H,W] or NULL for a black background. */
int mvp_composite_forward(int32_t N, int32_t H, int32_t W, const float *rayrgba, const float *ccw, const float *ccb,
                          const float *bg, float *irgbrec, float *rayalpha, void *stream);
/* Adjoint of the above.  grad_rayrgba [N,H,W,4] is written (not accumulated) contiguous channels-last, which is what
 * mvp_raymarch_backward takes.  grad_ccw / grad_ccb [N,3] (both or neither) are ACCUMULATED into: caller zero-fills;
 * grad_bg [N,3,H,W] is written.  rayrgba is needed only when grad_ccw or grad_bg is requested. */
int mvp_composite_backward(int32_t N, int32_t H, int32_t W, const float *rayrgba, const float *ccw, const float *bg,
                           const float *grad_irgbrec, const float *grad_rayalpha, float *grad_rayrgba, float *grad_ccw,
                           float *grad_ccb, float *grad_bg, void *stream);

/* Payload hand-off (SURVEY.md section 8f row 4).  tex [N, B*3, hb*B, wb*B] (channel d*3+c), opacity [N, B, hb*B, wb*B]
 * (channel d) -> tplate [N, hb*wb, B, B, B, 4] with
 *   tplate[n, i*wb+j, d, y, x, c<3] = relu(tex[n, d*3+c, i*B+y, j*B+x] * rgb_scale + rgb_bias),
 *   tplate[n, i*wb+j, d, y, x, 3]   = relu(opacity[n, d, i*B+y, j*B+x]).
 * The reference hard-codes rgb_scale = 25, rgb_bias = 100 (assembler.py:261).  1 <= B <= 64. */
int mvp_assemble_payload_forward(int32_t N, int32_t hb, int32_t wb, int32_t B, const float *tex, const float *opacity,
                                 float rgb_scale, float rgb_bias, float *tplate, void *stream);
/* Adjoint: grad_tex / grad_opacity (same shapes as tex / opacity) are written; `tplate` is the forward output (relu mask). */
int mvp_assemble_payload_backward(int32_t N, int32_t hb, int32_t wb, int32_t B, const float *tplate, const float *grad_tplate,
                                  float rgb_scale, float *grad_tex, float *grad_opacity, void *stream);

/* One subject's primitives materialised per view (what the decoders' batch dimension is in models/autoencoder.py:214-233
 * when all items of a batch show the same subject): dst[v, i] = src[i] for v < n_views, i < count floats.  One pass of
 * streaming 16-byte stores (scalar when count % 4 != 0 or a pointer is not 16-byte aligned); `expand().contiguous()` does the
 * same at a quarter of the rate.  count < 2^32 * 1024. */
int mvp_expand_views(const float *src, float *dst, size_t count, int32_t n_views, void *stream);
/* Its adjoint, and the local step of the per-subject gradient reduction (SURVEY.md section 8e: the views of a step share one
 * subject's primitives, their gradients are summed before the one all-reduce): dst[i] = sum over v < n_views of src[v, i], added
 * in view order (deterministic), one pass over the per-view gradients.  Same alignment rule as mvp_expand_views; n_views >= 1. */
int mvp_sum_views(const float *src, float *dst, size_t count, int32_t n_views, void *stream);

/* Test / diagnostics helper (host only, no device work): given a HOST copy of a workspace that a gradient-mode forward
 * has filled, counts the tiles whose slab list the forward saved for the backward (`saved`, lists with >= 1 entry) and the
 * tiles it had to mark not-saved because the list storage was full (`not_saved`; the backward rebuilds those). */
int mvp_debug_saved_tiles(const mvp_shape *shape, const void *host_workspace_copy, int *saved, int *not_saved);
/* Diagnostics builds only (-DMVP_TILE_CLOCKS=1, scripts/tile_clocks.py): byte offset of the per-tile clock records in the workspace. */
size_t mvp_debug_tileclk_offset(const mvp_shape *shape);

/* Number of kernels the last forward / backward call of this shape launches (for bench.py's gpu_launches). */
int mvp_forward_launch_count(uint32_t flags);
int mvp_backward_launch_count(uint32_t flags);

#ifdef __cplusplus
}
#endif
#endif /* MVPRAYMARCH_B200_H_ */
