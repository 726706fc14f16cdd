"""bfloat16 payloads (C-ABI MVP_FLAG_TPLATE_BF16) on the CPU emulation of the product kernels, and the flag's argument checks.

A bf16 value converts to fp32 exactly, so the kernels that read a bf16 template must render exactly what the fp32 kernels render
from its fp32 expansion: images and saturation colours bit for bit, gradients (fp32 in both cases) up to the order of the atomic
additions."""
import ctypes

import numpy as np
import pytest
import torch

from tests.helpers import build_case, relerr, scene_args_np

GRAD_TOL = 1e-6


def bf16_pair(x):
    """(bfloat16 bit patterns as uint16, their fp32 values) of an fp32 array: the top half of each float."""
    bits = (np.ascontiguousarray(x, np.float32).view(np.uint32) >> 16).astype(np.uint16)
    return bits, (bits.astype(np.uint32) << 16).view(np.float32)


def forward_backward_bf16(raypos, raydir, stepsize, tminmax, primpos, primrot, primscale, template, grad_rayrgba=None, warp=None,
                          fadescale=8.0, fadeexp=8.0, fwd_flags=0, bwd_flags=0, planes=False, order=None, clear_in_forward=False,
                          camera=None):
    """tests.emul.kernels.forward_backward for a template of bfloat16 bit patterns (uint16 [N,K,TD,TH,TW,4]): the same emulated
    calls with MVP_FLAG_TPLATE_BF16 set in both, the template's gradient in fp32 buffers.  Same arguments and return value."""
    from ava256_b200 import lib as abi
    from tests.emul.kernels import _aligned, _f32, _nan_like16, _p, load
    L = load()
    assert template.dtype == np.uint16
    template = np.ascontiguousarray(template)
    fwd_flags, bwd_flags = fwd_flags | abi.FLAG_TPLATE_BF16, bwd_flags | abi.FLAG_TPLATE_BF16
    primpos, primrot, primscale = map(_f32, (primpos, primrot, primscale))
    warp = None if warp is None else _f32(warp)
    cam = None
    if camera is not None:
        camarrs = [_f32(x) for x in camera[:4]]
        cam = abi.Camera(_p(camarrs[0]), _p(camarrs[1]), _p(camarrs[2]), _p(camarrs[3]), float(camera[4]), 0)
        N, H, W = camarrs[0].shape[0], int(camera[5]), int(camera[6])
    else:
        raypos, raydir, tminmax = map(_f32, (raypos, raydir, tminmax))
        N, H, W = raypos.shape[:3]
    shape = abi.Shape(N, H, W, primpos.shape[1], *template.shape[2:5])
    wsb = L.mvp_workspace_bytes(ctypes.byref(shape))
    ws = _aligned(wsb)
    want_grad = grad_rayrgba is not None
    rayrgba = np.full((N, H, W, 4), np.nan, np.float32)
    rgb_p = np.full((N, 3, H, W), np.nan, np.float32) if planes else None
    alpha_p = np.full((N, 1, H, W), np.nan, np.float32) if planes else None
    raysat = np.full((N, H, W, 3), np.nan, np.float32) if want_grad else None
    rayaux = np.zeros((N, H, W, 4), np.int32) if want_grad else None
    order = None if order is None else np.ascontiguousarray(order, dtype=np.int32)
    f32_shapes = [x.shape for x in (primpos, primrot, primscale)] + [template.shape]

    def common(s, flags):
        s.shape, s.stepsize, s.fadescale, s.fadeexp, s.flags = shape, float(stepsize), float(fadescale), float(fadeexp), flags
        s.raypos, s.raydir, s.tminmax = _p(raypos), _p(raydir), _p(tminmax)
        if cam is not None:
            s.camera = cam
        s.primpos, s.primrot, s.primscale, s.tplate = _p(primpos), _p(primrot), _p(primscale), _p(template)
        s.order = _p(order)
        s.workspace, s.workspace_bytes = _p(ws), wsb
        s.algo = 1 if warp is not None else 0
        if warp is not None:
            s.warp = _p(warp)
            s.WD, s.WH, s.WW = warp.shape[2:5]

    a = abi.ForwardArgs()
    common(a, fwd_flags)
    a.rayrgba, a.raysat, a.rayaux = (None if planes else _p(rayrgba)), _p(raysat), _p(rayaux)
    if planes:
        a.rayrgb_nchw, a.rayalpha_nchw = _p(rgb_p), _p(alpha_p)
    pre = None
    if clear_in_forward:
        pre = [_nan_like16(np.empty(sh, np.float32)) for sh in f32_shapes] + [_nan_like16(warp) if warp is not None else None]
        a.clear_grad_primpos, a.clear_grad_primrot, a.clear_grad_primscale, a.clear_grad_tplate = (_p(g) for g in pre[:4])
        a.clear_grad_warp = _p(pre[4])
    assert L.mvp_raymarch_forward(ctypes.byref(a), None) == 0
    if pre is not None:
        assert all(g is None or not g.any() for g in pre), "the forward must leave the clear_grad_* buffers zero"
    if planes:
        rayrgba = np.ascontiguousarray(np.concatenate([rgb_p, alpha_p], axis=1).transpose(0, 2, 3, 1))
    if not want_grad:
        return rayrgba, None, None
    grad_rayrgba = _f32(grad_rayrgba)
    fill = np.nan if (bwd_flags & abi.FLAG_ZERO_GRADS) else 0.0
    grads = pre[:4] if pre is not None else [np.full(sh, fill, np.float32) for sh in f32_shapes]
    gwarp = pre[4] if pre is not None else (np.full_like(warp, fill) if warp is not None else None)
    b = abi.BackwardArgs()
    common(b, abi.FLAG_ACCEL_VALID | bwd_flags)
    if planes:
        g_rgb = np.ascontiguousarray(grad_rayrgba.transpose(0, 3, 1, 2)[:, :3])
        g_alpha = np.ascontiguousarray(grad_rayrgba.transpose(0, 3, 1, 2)[:, 3:4])
        b.grad_rayrgb_nchw, b.grad_rayalpha_nchw = _p(g_rgb), _p(g_alpha)
    b.grad_rayrgba, b.raysat, b.rayaux = (None if planes else _p(grad_rayrgba)), _p(raysat), _p(rayaux)
    b.grad_primpos, b.grad_primrot, b.grad_primscale, b.grad_tplate = (_p(g) for g in grads)
    if warp is not None:
        b.grad_warp = _p(gwarp)
    assert L.mvp_raymarch_backward(ctypes.byref(b), None) == 0
    return rayrgba, raysat, grads + ([gwarp] if gwarp is not None else [])


@pytest.fixture()
def kernels():
    from tests.emul import kernels as k
    k.use_variant(())
    k.load()
    yield k
    k.set_lane_order("forward")
    k.use_variant(())


def assert_same_render(ref, got):
    out0, sat0, g0 = ref
    out1, sat1, g1 = got
    assert np.array_equal(out0, out1)
    assert (sat0 is None) == (sat1 is None)
    if sat0 is not None:
        assert np.array_equal(sat0, sat1)
    if g0 is not None:
        assert len(g0) == len(g1)
        for nm, x, y in zip(("primpos", "primrot", "primscale", "template", "warp"), g0, g1):
            assert y.dtype == np.float32 and y.shape == x.shape, nm
            assert np.isfinite(y).all() and relerr(y, x) <= GRAD_TOL, nm


def run_pair(kernels, a, **kw):
    """The same call with the fp32 expansion of a bf16 template and with the bf16 template itself."""
    bits, f32 = bf16_pair(a[7])
    a32, a16 = list(a), list(a)
    a32[7], a16[7] = f32, bits
    return kernels.forward_backward(*a32, **kw), forward_backward_bf16(*a16, **kw)


@pytest.mark.parametrize("name", ["tiny", "head_small", "noncubic", "many_overlaps", "warp_small", "gradcheck_ragged"])
def test_bf16_template_renders_like_its_fp32_expansion(kernels, name):
    s, grad = build_case(name)
    a, kw = scene_args_np(s)
    ref, got = run_pair(kernels, a, grad_rayrgba=grad.numpy(), **kw)
    assert float(ref[0][..., 3].max()) > 0.0
    assert_same_render(ref, got)
    ref, got = run_pair(kernels, a, **kw)                       # inference kernels (no raysat / rayaux)
    assert_same_render(ref, got)


def test_bf16_template_shared_primitives(kernels):
    """MVP_FLAG_SHARED_PRIMS with a bf16 [1,K,...] template."""
    from ava256_b200 import lib, scene
    s, _ = build_case("head_small")
    N, H, W = 3, s["raypos"].shape[1], s["raypos"].shape[2]
    rp, rd, tmm = scene.make_rays(N, H, W, view_offset=2)
    g = torch.randn(N, H, W, 4, generator=torch.Generator().manual_seed(2)).numpy()
    a = [rp.numpy(), rd.numpy(), s["stepsize"], tmm.numpy()] + [s[k][:1].numpy() for k in ("primpos", "primrot", "primscale", "template")]
    ref, got = run_pair(kernels, a, grad_rayrgba=g, fadescale=s["fadescale"], fadeexp=s["fadeexp"], fwd_flags=lib.FLAG_SHARED_PRIMS,
                        bwd_flags=lib.FLAG_SHARED_PRIMS | lib.FLAG_ZERO_GRADS)
    assert float(ref[0][..., 3].max()) > 0.05 and got[2][3].shape[0] == 1
    assert_same_render(ref, got)


@pytest.mark.parametrize("planes", [False, True])
def test_bf16_template_camera_rays(kernels, planes):
    """Rays generated in the kernels from the camera (mvp_camera), with channels-last or image-plane outputs."""
    from ava256_b200 import scene
    n, H, W, K, T = 2, 64, 42, 64, 8
    viewpos, viewrot, focal, princpt = scene.make_cameras(n, H, W, view_offset=3)
    s = scene.make_scene(n, H, W, K, T, view_offset=3, alpha_mu=1.0, alpha_sigma=2.0, share_primitives=False)
    g = torch.randn(n, H, W, 4, generator=torch.Generator().manual_seed(5)).numpy()
    a = [None, None, 1.0 / 64, None] + [s[k].numpy() for k in ("primpos", "primrot", "primscale", "template")]
    cam = (viewpos.numpy(), viewrot.numpy(), focal.numpy(), princpt.numpy(), scene.VOLRADIUS, H, W)
    ref, got = run_pair(kernels, a, grad_rayrgba=g, planes=planes, camera=cam)
    assert float(ref[0][..., 3].max()) > 0.05
    assert_same_render(ref, got)


def test_bf16_template_tiny_lists_and_library_zero_fill(kernels):
    """MVP_FLAG_TEST_TINY_LISTS (most tiles take the backward's rebuild path) and MVP_FLAG_ZERO_GRADS (NaN-filled gradient buffers
    that the library zero-fills)."""
    from ava256_b200 import lib
    s, grad = build_case("head_small")
    a, kw = scene_args_np(s)
    ref, got = run_pair(kernels, a, grad_rayrgba=grad.numpy(), fwd_flags=lib.FLAG_TEST_TINY_LISTS, bwd_flags=lib.FLAG_ZERO_GRADS, **kw)
    loaded, rebuilt = ctypes.c_int(), ctypes.c_int()
    kernels.load().mvp_emul_saved_list_tiles(ctypes.byref(loaded), ctypes.byref(rebuilt))
    assert rebuilt.value > 0
    assert_same_render(ref, got)


@pytest.mark.parametrize("name", ["head_small", "warp_head"])
def test_bf16_template_forward_clears_fp32_gradient_buffers(kernels, name):
    """clear_grad_tplate is an fp32 buffer also for a bf16 template: the gradient-mode forward zero-fills all of it."""
    s, grad = build_case(name)
    a, kw = scene_args_np(s)
    ref, got = run_pair(kernels, a, grad_rayrgba=grad.numpy(), clear_in_forward=True, **kw)
    assert_same_render(ref, got)


def test_bf16_template_marching_order(kernels):
    """An explicit marching order (usebvh=True) with a bf16 template."""
    from ava256_b200.op import morton_order
    s, grad = build_case("gradcheck_ragged")
    a, kw = scene_args_np(s)
    order = morton_order(s["primpos"]).numpy().astype(np.int32)[:, ::-1].copy()
    ref, got = run_pair(kernels, a, grad_rayrgba=grad.numpy(), order=order, **kw)
    assert_same_render(ref, got)


def test_bf16_template_needs_8_byte_alignment_only(kernels):
    """A bf16 template that starts 8 bytes past a 16-byte boundary is a valid argument and renders the same."""
    s, grad = build_case("gradcheck_ragged")
    a, kw = scene_args_np(s)
    bits, _ = bf16_pair(a[7])
    raw = np.zeros(bits.size + 16, np.uint16)
    off = ((-raw.ctypes.data) % 16) // 2 + 4                   # 8 bytes past a 16-byte boundary
    shifted = raw[off:off + bits.size].reshape(bits.shape)
    shifted[...] = bits
    assert shifted.ctypes.data % 16 == 8
    a16 = list(a)
    a16[7] = bits
    ref = forward_backward_bf16(*a16, grad_rayrgba=grad.numpy(), **kw)
    a16[7] = shifted
    got = forward_backward_bf16(*a16, grad_rayrgba=grad.numpy(), **kw)
    assert_same_render(ref, got)


# ------------------------------------------------------------------------------------------------------------------
# the flag at the C-ABI, without a device: every check below returns before any device work
# ------------------------------------------------------------------------------------------------------------------
def _args(cls, fields):
    from ava256_b200 import lib
    a = cls()
    a.shape = lib.Shape(1, 8, 8, 4, 2, 2, 2)
    a.stepsize = 0.1
    for f in fields:
        setattr(a, f, ctypes.c_void_p(256))
    a.workspace_bytes = 1 << 30
    return a


def test_supported_flags_include_bf16_template():
    from ava256_b200 import lib
    flags = lib.LIB.mvp_supported_flags()
    assert lib.FLAG_TPLATE_BF16 == 8
    for f in (lib.FLAG_ACCEL_VALID, lib.FLAG_ZERO_GRADS, lib.FLAG_SHARED_PRIMS, lib.FLAG_TPLATE_BF16):
        assert flags & f, f


def test_bf16_template_alignment_is_checked():
    from ava256_b200 import lib
    fwd = ("raypos", "raydir", "tminmax", "primpos", "primrot", "primscale", "tplate", "rayrgba", "workspace")
    bwd = ("raypos", "raydir", "tminmax", "primpos", "primrot", "primscale", "tplate", "grad_rayrgba", "raysat", "rayaux",
           "grad_primpos", "grad_primrot", "grad_primscale", "grad_tplate", "workspace")
    for cls, fields, call in ((lib.ForwardArgs, fwd, lib.LIB.mvp_raymarch_forward), (lib.BackwardArgs, bwd, lib.LIB.mvp_raymarch_backward)):
        a = _args(cls, fields)
        a.flags = lib.FLAG_TPLATE_BF16
        a.tplate = ctypes.c_void_p(256 + 4)                      # 4 bytes off 8-byte alignment
        assert call(ctypes.byref(a), None) == -6                 # MVP_ERR_ALIGN
        a.flags = 0
        a.tplate = ctypes.c_void_p(256 + 8)                      # fp32 voxels need 16 bytes
        assert call(ctypes.byref(a), None) == -6
    a = _args(lib.BackwardArgs, bwd)
    a.flags = lib.FLAG_TPLATE_BF16
    a.grad_tplate = ctypes.c_void_p(256 + 8)                     # the gradient stays fp32: 16 bytes
    assert lib.LIB.mvp_raymarch_backward(ctypes.byref(a), None) == -6
    assert b"bf16" in lib.LIB.mvp_error_string(-6)


def test_op_checks_device_before_dtype():
    """Host tensors raise the CUDA error first, whatever their dtype (bf16 and fp16 alike)."""
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    s, _ = build_case("gradcheck_ragged")
    for dt in (torch.bfloat16, torch.float16):
        with pytest.raises(RuntimeError, match="CUDA"):
            mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (s["primpos"], s["primrot"], s["primscale"]),
                        s["template"].to(dt), None)
