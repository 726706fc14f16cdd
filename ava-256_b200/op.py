"""torch.autograd front-end of the B200 raymarcher: the host-side mirror of the reference's op
(/root/reference/extensions/mvpraymarch/mvpraymarch.py:87-390) on top of the C-ABI in include/mvpraymarch_b200.h.

Same contract as the reference: fp32 CUDA tensors (template and primitive transforms may also be bf16, as decoders produce
them under torch.autocast), contiguous, caller-visible output rayrgba [N,H,W,4] that
participates in autograd with gradients for primpos, primrot, primscale, template and (algo 1) warp, None for
everything else (mvpraymarch.py:279-292).  Differences that are deliberate:
  * kernels run on torch's current stream (the reference launches on legacy stream 0, mvpraymarch.cpp:277);
  * no allocation or sync inside the native call (the reference cudaMalloc/cudaFree's per forward, bvh.cu:261-293);
  * the acceleration structure is a screen-space bucket list, not the BVH tensors of build_accel (:21-84);
    it is kept for backward instead of being rebuilt;
  * 64-bit indexing (the reference overflows int32 at N*K*T^3*4 >= 2^31, primsampler.h:31-36).
"""
import ctypes

import torch
from torch.autograd import Function

from . import lib as _lib


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _aligned(t, nbytes):
    """The kernels read channels-last buffers with 128-bit accesses (C-ABI: MVP_ERR_ALIGN).  A contiguous view into a
    larger buffer can start anywhere; such a tensor is copied once to a fresh (256-byte aligned) allocation."""
    if t is not None and t.data_ptr() % nbytes:
        return t.clone()
    return t


_F32 = (torch.float32,)
# What decoders produce under torch.autocast(dtype=torch.bfloat16).  A bf16 template is read as bf16 by the kernels (C-ABI
# MVP_FLAG_TPLATE_BF16); bf16 primitive transforms (K*60 bytes per view) are converted to fp32 here.
_F32_BF16 = (torch.float32, torch.bfloat16)


def _check_f32_cuda(name, t, dtypes=_F32):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor" % name)          # mvpraymarch.cpp:102
    if not t.is_contiguous():
        raise RuntimeError("%s must be contiguous" % name)             # mvpraymarch.cpp:103
    if t.dtype not in dtypes:
        raise RuntimeError("%s must be %s" % (name, " or ".join(str(d)[len("torch."):] for d in dtypes)))


class MVPRaymarch(Function):
    """Custom Function for raymarching Mixture of Volumetric Primitives (reference: mvpraymarch.py:87-292)."""

    @staticmethod
    def forward(ctx, raypos, raydir, stepsize, tminmax, primpos, primrot, primscale, template, warp, rayterm,
                gradmode, options):
        algo = options["algo"]
        if algo not in (0, 1):
            raise NotImplementedError("mvpraymarch_b200: algo must be 0 or 1 (the reference launches nothing for other "
                                      "values, mvpraymarch_kernel.cu:104-105)")
        if algo == 1 and warp is None:
            raise RuntimeError("mvpraymarch_b200: algo=1 samples a warp field (PrimSamplerTW<true>); pass `warp`")
        if options["usebvh"] is False:
            raise NotImplementedError("mvpraymarch_b200: usebvh=False passes a null BVH to the reference kernels "
                                      "(mvpraymarch.py:132-134) and is not a usable mode there either")
        camera = options.get("_camera")        # (viewpos, viewrot, focal, princpt, volradius, H, W): rays generated in the kernels
        if camera is not None:
            assert raypos is None and raydir is None and tminmax is None
            viewpos, viewrot, focal, princpt, volradius, camH, camW = camera
            for name, t, tail in (("viewpos", viewpos, (3,)), ("viewrot", viewrot, (3, 3)), ("focal", focal, (2,)), ("princpt", princpt, (2,))):
                _check_f32_cuda(name, t)                                  # utils.py:24-25 / utils.cpp CHECK_CUDA
                assert t.shape == (viewpos.size(0),) + tail, "%s must be [N,%s]" % (name, ",".join(map(str, tail)))
                assert t.device == primpos.device, "%s must be on the primitives' device" % name
            assert int(camH) >= 1 and int(camW) >= 1 and float(volradius) > 0.0
        else:
            # same shape contract as mvpraymarch.py:112-127
            assert raypos.is_contiguous() and raypos.size(3) == 3
            assert raydir.is_contiguous() and raydir.size(3) == 3
            assert tminmax.is_contiguous() and tminmax.size(3) == 2
        assert primpos.is_contiguous() and primpos.size(2) == 3
        assert primrot.is_contiguous() and primrot.size(2) == 3
        assert primscale.is_contiguous() and primscale.size(2) == 3
        assert template.is_contiguous() and template.dim() == 6 and template.size(-1) == 4, \
            "channels-last template [N,K,TD,TH,TW,4] required (the reference sampler is always channels-last, primsampler.h:16)"
        for name, t in (("raypos", raypos), ("raydir", raydir), ("tminmax", tminmax)):
            if t is not None:
                _check_f32_cuda(name, t)
        for name, t in (("primpos", primpos), ("primrot", primrot), ("primscale", primscale), ("template", template)):
            _check_f32_cuda(name, t, _F32_BF16)
        if warp is not None:                                           # mvpraymarch.py:124
            assert warp.is_contiguous() and warp.dim() == 6 and warp.size(-1) == 3, \
                "channels-last warp field [N,K,WD,WH,WW,3] required"
            _check_f32_cuda("warp", warp)
        usewarp = algo == 1                                            # algo 0 ignores a warp field, like the reference
        # bf16 primitive transforms are rendered (and differentiated) in fp32; their gradients go back in the input dtype
        prim_dtypes = (primpos.dtype, primrot.dtype, primscale.dtype)
        primpos, primrot, primscale = primpos.float(), primrot.float(), primscale.float()
        bf16 = template.dtype == torch.bfloat16

        if camera is not None:
            N, H, W = viewpos.size(0), int(camH), int(camW)
        else:
            N, H, W = raypos.shape[:3]
        K = primpos.size(1)
        TD, TH, TW = template.shape[2:5]
        dev = primpos.device
        # The reference never checks that the leading dimensions agree (a mismatch reads out of bounds there).  Here:
        # rays and tminmax must agree; the primitive tensors must agree with each other and have a batch of N, or of 1
        # = one set of primitives shared by all N views (extension, SURVEY.md section 8e "optional fast path":
        # nothing is replicated in HBM and the gradients of all views accumulate into the one set).
        if camera is None:
            assert raydir.shape[:3] == (N, H, W) and tminmax.shape[:3] == (N, H, W), "raypos / raydir / tminmax disagree on [N,H,W]"
        NP = primpos.size(0)
        assert NP in (N, 1), "primitive batch (%d) must equal the number of views (%d) or be 1 (shared)" % (NP, N)
        assert primrot.shape[:2] == (NP, K) and primscale.shape[:2] == (NP, K) and template.shape[:2] == (NP, K), \
            "primpos / primrot / primscale / template disagree on [N,K]"
        if warp is not None:
            assert warp.shape[:2] == (NP, K), "warp disagrees with the primitives on [N,K]"
        shared = NP == 1 and N > 1
        template, tminmax = _aligned(template, 8 if bf16 else 16), _aligned(tminmax, 8)
        with torch.cuda.device(dev):
            wsbytes = _lib.workspace_bytes(N, H, W, K, TD, TH, TW)
            workspace = torch.empty(wsbytes, dtype=torch.uint8, device=dev)
            planes = bool(options.get("_planes", False))   # image-plane outputs (MVPRaymarchPlanes below)
            if planes:
                rayrgba = None
                rayrgb = torch.empty((N, 3, H, W), dtype=torch.float32, device=dev)
                rayalpha = torch.empty((N, 1, H, W), dtype=torch.float32, device=dev)
            else:
                rayrgba = torch.empty((N, H, W, 4), dtype=torch.float32, device=dev)
            if gradmode:
                raysat = torch.empty((N, H, W, 3), dtype=torch.float32, device=dev)
                rayaux = torch.empty((N, H, W, 4), dtype=torch.int32, device=dev)
            else:
                raysat = rayaux = None
            a = _lib.ForwardArgs()
            a.shape = _lib.Shape(N, H, W, K, TD, TH, TW)
            a.stepsize, a.fadescale, a.fadeexp = float(stepsize), float(options["fadescale"]), float(options["fadeexp"])
            a.flags = (_lib.FLAG_SHARED_PRIMS if shared else 0) | (_lib.FLAG_TPLATE_BF16 if bf16 else 0)
            a.raypos, a.raydir, a.tminmax = _ptr(raypos), _ptr(raydir), _ptr(tminmax)
            if camera is not None:
                a.camera = _lib.Camera(_ptr(viewpos), _ptr(viewrot), _ptr(focal), _ptr(princpt), float(volradius), 0)
            a.primpos, a.primrot, a.primscale = _ptr(primpos), _ptr(primrot), _ptr(primscale)
            a.tplate = _ptr(template)
            a.rayrgba, a.raysat, a.rayaux = _ptr(rayrgba), _ptr(raysat), _ptr(rayaux)
            if planes:
                a.rayrgb_nchw, a.rayalpha_nchw = _ptr(rayrgb), _ptr(rayalpha)
            order = options.get("_order")                              # [NP,K] int32 marching order (usebvh=True) or None
            if order is not None:
                assert order.dtype == torch.int32 and order.is_contiguous() and tuple(order.shape) == (NP, K)
                a.order = _ptr(order)
            a.workspace, a.workspace_bytes = _ptr(workspace), wsbytes
            a.algo = 1 if usewarp else 0
            if usewarp:
                a.warp = _ptr(warp)
                a.WD, a.WH, a.WW = warp.shape[2:5]
            grads = None
            if gradmode:
                # The gradient buffers of the backward (mvpraymarch.py:240-246 zeros_like's them there) are made now and zero-filled
                # by the forward's render kernel on the side (mvp_forward_args::clear_grad_*): no memset pass in the step.
                # The template's gradient is accumulated in fp32 also for a bf16 template.
                grads = [torch.empty_like(primpos), torch.empty_like(primrot), torch.empty_like(primscale),
                         torch.empty_like(template, dtype=torch.float32), torch.empty_like(warp) if usewarp else None]
                a.clear_grad_primpos, a.clear_grad_primrot, a.clear_grad_primscale = _ptr(grads[0]), _ptr(grads[1]), _ptr(grads[2])
                a.clear_grad_tplate, a.clear_grad_warp = _ptr(grads[3]), _ptr(grads[4])
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.LIB.mvp_raymarch_forward(ctypes.byref(a), ctypes.c_void_p(stream)))

        if gradmode:
            ctx.grads = grads
            ctx.save_for_backward(raypos, raydir, tminmax, primpos, primrot, primscale, template, raysat, rayaux, workspace, warp)
            ctx.camera = camera                # camera tensors are plain inputs without gradients (utils.py:45-46 returns None for all)
            ctx.nhw = (N, H, W)
            ctx.order = order
            ctx.options = options
            ctx.stepsize = float(stepsize)
            ctx.shared = shared
            ctx.prim_dtypes = prim_dtypes
        if planes:
            return rayrgb, rayalpha
        return rayrgba

    @staticmethod
    def backward(ctx, grad_rayrgba, grad_rayalpha=None):
        """grad_rayrgba [N,H,W,4]; or, for MVPRaymarchPlanes, (grad_rayrgb [N,3,H,W], grad_rayalpha [N,1,H,W])."""
        raypos, raydir, tminmax, primpos, primrot, primscale, template, raysat, rayaux, workspace, warp = ctx.saved_tensors
        options = ctx.options
        N, H, W = ctx.nhw
        K = primpos.size(1)
        TD, TH, TW = template.shape[2:5]
        dev = primpos.device
        with torch.cuda.device(dev):
            planes = bool(options.get("_planes", False))
            if planes:
                grad_rgb = grad_rayrgba.contiguous() if grad_rayrgba is not None else torch.zeros((N, 3, H, W), device=dev)
                grad_alpha = grad_rayalpha.contiguous() if grad_rayalpha is not None else torch.zeros((N, 1, H, W), device=dev)
                grad_rayrgba = None
            else:
                grad_rayrgba = _aligned(grad_rayrgba.contiguous(), 16)     # mvpraymarch.py:264
            usewarp = options["algo"] == 1
            grads, ctx.grads = ctx.grads, None
            fresh = grads is not None          # the forward's render kernel zero-filled them; a second backward through the
            if not fresh:                      # same graph (retain_graph) gets new ones, zero-filled by the library
                grads = [torch.empty_like(primpos), torch.empty_like(primrot), torch.empty_like(primscale),
                         torch.empty_like(template, dtype=torch.float32), torch.empty_like(warp) if usewarp else None]
            grad_primpos, grad_primrot, grad_primscale, grad_template, grad_warp = grads
            del grads
            if warp is not None and not usewarp:                       # mvpraymarch.py:246 (zero when algo 0 ignores it)
                grad_warp = torch.zeros_like(warp)
            bf16 = template.dtype == torch.bfloat16
            a = _lib.BackwardArgs()
            a.shape = _lib.Shape(N, H, W, K, TD, TH, TW)
            a.stepsize, a.fadescale, a.fadeexp = ctx.stepsize, float(options["fadescale"]), float(options["fadeexp"])
            a.flags = _lib.FLAG_ACCEL_VALID | (0 if fresh else _lib.FLAG_ZERO_GRADS) | (_lib.FLAG_SHARED_PRIMS if ctx.shared else 0) | \
                (_lib.FLAG_TPLATE_BF16 if bf16 else 0)
            a.raypos, a.raydir, a.tminmax = _ptr(raypos), _ptr(raydir), _ptr(tminmax)
            if ctx.camera is not None:
                viewpos, viewrot, focal, princpt, volradius = ctx.camera[:5]
                a.camera = _lib.Camera(_ptr(viewpos), _ptr(viewrot), _ptr(focal), _ptr(princpt), float(volradius), 0)
            a.primpos, a.primrot, a.primscale = _ptr(primpos), _ptr(primrot), _ptr(primscale)
            a.tplate = _ptr(template)
            a.grad_rayrgba, a.raysat, a.rayaux = _ptr(grad_rayrgba), _ptr(raysat), _ptr(rayaux)
            if planes:
                a.grad_rayrgb_nchw, a.grad_rayalpha_nchw = _ptr(grad_rgb), _ptr(grad_alpha)
            if ctx.order is not None:
                a.order = _ptr(ctx.order)
            a.grad_primpos, a.grad_primrot, a.grad_primscale = _ptr(grad_primpos), _ptr(grad_primrot), _ptr(grad_primscale)
            a.grad_tplate = _ptr(grad_template)
            a.workspace, a.workspace_bytes = _ptr(workspace), workspace.numel()
            a.algo = 1 if usewarp else 0
            if usewarp:
                a.warp, a.grad_warp = _ptr(warp), _ptr(grad_warp)
                a.WD, a.WH, a.WW = warp.shape[2:5]
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.LIB.mvp_raymarch_backward(ctypes.byref(a), ctypes.c_void_p(stream)))
            if bf16:                           # one round-to-nearest-even pass; the fp32 accumulator is freed here
                grad_template = grad_template.to(torch.bfloat16)
            pd = ctx.prim_dtypes
            grad_primpos, grad_primrot, grad_primscale = grad_primpos.to(pd[0]), grad_primrot.to(pd[1]), grad_primscale.to(pd[2])
        return (None, None, None, None, grad_primpos, grad_primrot, grad_primscale, grad_template, grad_warp, None, None, None)


class MVPRaymarchPlanes(MVPRaymarch):
    """Same op with the outputs as the caller uses them: (rayrgb [N,3,H,W], rayalpha [N,1,H,W]), written by the render
    kernel's epilogue, and the gradient taken as those two planes by the backward's prologue -- the permute + two
    `.contiguous()` copies of models/raymarchers/mvpraymarcher.py:50-51 and the `.contiguous()` of the incoming gradient
    (mvpraymarch.py:264) never run (SURVEY.md section 8f row 2)."""

    @staticmethod
    def forward(ctx, raypos, raydir, stepsize, tminmax, primpos, primrot, primscale, template, warp, rayterm, gradmode, options):
        options = dict(options, _planes=True)
        return MVPRaymarch.forward(ctx, raypos, raydir, stepsize, tminmax, primpos, primrot, primscale, template, warp, rayterm,
                                   gradmode, options)

    @staticmethod
    def backward(ctx, grad_rayrgb, grad_rayalpha):
        return MVPRaymarch.backward(ctx, grad_rayrgb, grad_rayalpha)


def morton_codes(primpos):
    """30-bit Morton codes of the primitive centres, normalised per view to their bounding box: the reference's
    build_accel (mvpraymarch.py:46-53) + morton3D / expand_bits (bvh.cu:20-41).  [N,K] int64."""
    cmax = primpos.max(dim=1, keepdim=True)[0]
    cmin = primpos.min(dim=1, keepdim=True)[0]
    c = (primpos - cmin) / (cmax - cmin).clamp(min=1e-8)                       # mvpraymarch.py:50
    q = (c * 1024.0).clamp(0.0, 1023.0).to(torch.int64)                        # bvh.cu:33-35, (unsigned int) truncates

    def expand_bits(v):                                                        # bvh.cu:22-28 (uint32 arithmetic)
        v = (v * 0x00010001) & 0xFF0000FF
        v = (v * 0x00000101) & 0x0F00F00F
        v = (v * 0x00000011) & 0xC30C30C3
        v = (v * 0x00000005) & 0x49249249
        return v

    return expand_bits(q[..., 0]) * 4 + expand_bits(q[..., 1]) * 2 + expand_bits(q[..., 2])   # bvh.cu:39


def morton_codes_native(primpos):
    """The same codes from the library's kernel (`mvp_compute_morton`, the reference's compute_morton): the normalisation to the
    bounding box stays in torch like in the reference (mvpraymarch.py:46-50).  [N,K] int32."""
    p = primpos.detach().float()
    cmax = p.max(dim=1, keepdim=True)[0]
    cmin = p.min(dim=1, keepdim=True)[0]
    c = ((p - cmin) / (cmax - cmin).clamp(min=1e-8)).contiguous()
    code = torch.empty(p.shape[:2], dtype=torch.int32, device=p.device)
    with torch.cuda.device(p.device):
        _lib.check(_lib.LIB.mvp_compute_morton(p.shape[0], p.shape[1], _ptr(c), _ptr(code),
                                               ctypes.c_void_p(torch.cuda.current_stream(p.device).cuda_stream)))
    return code


def morton_order(primpos):
    """sortedobjid [N,K] (int64): primitive indices in ascending Morton code (mvpraymarch.py:54-55).  Ties keep index
    order (stable), where the reference's torch.sort leaves them unspecified."""
    codes = morton_codes_native(primpos) if primpos.is_cuda else morton_codes(primpos.detach())
    return torch.sort(codes, dim=-1, stable=True)[1]


def _take(t, order):
    """t[n, order[n, k], ...] (differentiable)."""
    if t is None:
        return None
    idx = order.view(order.shape + (1,) * (t.dim() - 2)).expand(order.shape + tuple(t.shape[2:]))
    return torch.gather(t, 1, idx)


def mvpraymarch(
    raypos,
    raydir,
    stepsize,
    tminmax,
    primtransf,
    template,
    warp,
    rayterm=None,
    algo=0,
    usebvh="fixedorder",
    sortprims=False,
    randomorder=False,
    maxhitboxes=512,
    synchitboxes=True,
    chlast=True,
    fadescale=8.0,
    fadeexp=8.0,
    accum=0,
    termthresh=0.0,
    griddim=3,
    blocksize=(8, 16),
    bwdblocksize=(8, 16),
):
    """Drop-in for extensions.mvpraymarch.mvpraymarch.mvpraymarch (reference mvpraymarch.py:295-390).

    Same parameters, same defaults.  `sortprims`, `randomorder`, `maxhitboxes`, `synchitboxes`, `chlast`, `accum`,
    `termthresh`, `griddim`, `blocksize`, `bwdblocksize` and `rayterm` are accepted and, exactly like in the
    reference kernels (SURVEY.md section 8a, "accepted but ignored"), have no effect on the result.

    `usebvh="fixedorder"` (default) marches the primitives of a tile in index order.  `usebvh=True` marches them in
    Morton order of their centres -- the order the reference's LBVH branch computes (`sortedobjid`, mvpraymarch.py:46-55)
    but its kernels never apply (they hard-code the implicit heap, utils.h:740-742; SURVEY.md section 2.3 K5): codes from the
    library's `mvp_compute_morton`, one `torch.sort`, and the order goes to the kernels as an indirection (no tensor is
    gathered or copied).  The order only matters for rays that saturate.
    Returns rayrgba [N,H,W,4]."""
    if usebvh is False:
        raise NotImplementedError("mvpraymarch_b200: usebvh=False hands the reference kernels a null BVH "
                                  "(mvpraymarch.py:132-134); use 'fixedorder' or True")
    if isinstance(primtransf, tuple):
        primpos, primrot, primscale = primtransf
    else:                                                              # packed [N,K,5,3]  (mvpraymarch.py:353-360)
        primpos = primtransf[:, :, 0, :].contiguous()
        primrot = primtransf[:, :, 1:4, :].contiguous()
        primscale = primtransf[:, :, 4, :].contiguous()
    order = None
    if usebvh != "fixedorder":
        # Morton order of the centres as an indirection inside the kernels (C-ABI `order`): nothing is gathered or copied
        order = morton_order(primpos).to(torch.int32).contiguous()
    options = {
        "algo": algo, "usebvh": usebvh, "sortprims": sortprims, "randomorder": randomorder,
        "maxhitboxes": maxhitboxes, "synchitboxes": synchitboxes, "chlast": chlast, "fadescale": fadescale,
        "fadeexp": fadeexp, "accum": accum, "termthresh": termthresh, "griddim": griddim, "blocksize": blocksize,
        "bwdblocksize": bwdblocksize, "_order": order,
    }
    if _CAMERA.get("cam") is not None:
        options["_camera"] = _CAMERA["cam"]
    fn = MVPRaymarchPlanes if _PLANES.get("on") else MVPRaymarch
    return fn.apply(raypos, raydir, stepsize, tminmax, primpos, primrot, primscale, template, warp, rayterm,
                    torch.is_grad_enabled(), options)


_PLANES = {}
_CAMERA = {}


def mvpraymarch_planes(*args, **kwargs):
    """`mvpraymarch` with image-plane outputs: same parameters, returns (rayrgb [N,3,H,W], rayalpha [N,1,H,W]) instead of
    rayrgba [N,H,W,4] (see MVPRaymarchPlanes; used by `ava256_b200.raymarcher.Raymarcher`)."""
    _PLANES["on"] = True
    try:
        return mvpraymarch(*args, **kwargs)
    finally:
        _PLANES["on"] = False


def mvpraymarch_camera(viewpos, viewrot, focal, princpt, pixelcoords, volradius, stepsize, primtransf, template, warp, planes=False,
                       **kwargs):
    """`compute_raydirs` + `mvpraymarch` of models/autoencoder.py:240-252 as ONE call: the first six parameters are those of the
    reference's compute_raydirs (extensions/utils/utils.py:48-51), the rest those of `mvpraymarch` after its ray arguments.

    With `pixelcoords` given as the `(W, H)` tuple (the integer pixel grid, utils.py:28-30) the rays never exist in memory: the
    render kernels generate each tile's rays in their prologue from the camera (C-ABI `mvp_camera`), bit-identical to what
    `compute_raydirs` would have written -- 32 bytes per ray that are neither written by a generation pass nor read by forward
    and backward -- and the accel build takes the camera as it is instead of fitting one to the ray field.  With a `pixelcoords`
    tensor (arbitrary sample positions) the two calls are made one after the other, as in the reference.
    No gradients flow to the camera (the reference's compute_raydirs backward returns None for every input, utils.py:45-46).
    Returns rayrgba [N,H,W,4], or (rayrgb [N,3,H,W], rayalpha [N,1,H,W]) with planes=True."""
    march = mvpraymarch_planes if planes else mvpraymarch
    if not isinstance(pixelcoords, tuple):
        from .raydirs import compute_raydirs
        raypos, raydir, tminmax = compute_raydirs(viewpos, viewrot, focal, princpt, pixelcoords, volradius)
        return march(raypos, raydir, stepsize, tminmax, primtransf, template, warp, **kwargs)
    W, H = pixelcoords
    _CAMERA["cam"] = (viewpos, viewrot, focal, princpt, float(volradius), int(H), int(W))
    try:
        return march(None, None, stepsize, None, primtransf, template, warp, **kwargs)
    finally:
        _CAMERA["cam"] = None
