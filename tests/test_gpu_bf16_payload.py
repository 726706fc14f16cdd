"""GPU tests of bfloat16 payloads: `mvpraymarch(..., template_bf16)` against `mvpraymarch(..., template_bf16.float())`.

The kernels convert each bf16 voxel to fp32 on load, which is exact, so the image must be bit-identical to the fp32 op's on the
upcast template.  The template's gradient is accumulated in fp32 and rounded to bf16 once, so it must equal the fp32 op's
gradient rounded to bf16 up to one bf16 ulp (plus the fp32 atomic-order noise both runs carry).  bf16 primitive transforms are
converted to fp32 by the op; their gradients come back in bf16."""
import pytest
import torch

from tests.helpers import CASES, SAMPLED_CASES, build_case

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
PRIMS = ("primpos", "primrot", "primscale")
ATOMIC_TOL = 1e-5          # fp32 gradients of two runs differ by the order of their atomic additions only


def _trelerr(a, b):
    return float((a.float() - b.float()).abs().max()) / max(float(b.float().abs().max()), 1e-30)


def _assert_within_bf16_ulp(got, ref32):
    """got (bf16) == ref32 (fp32) rounded to bf16, to one bf16 ulp of the larger magnitude, plus the atomic-order allowance."""
    assert got.dtype == BF16 and got.shape == ref32.shape
    want = ref32.to(BF16).float()
    g = got.float()
    _, e = torch.frexp(torch.maximum(g.abs(), want.abs()))
    ulp = torch.ldexp(torch.ones_like(g), e - 8)                 # bf16: 8 significant bits
    slack = ATOMIC_TOL * float(ref32.abs().max())
    assert bool(torch.isfinite(g).all())
    assert bool(((g - want).abs() <= ulp + slack).all()), float(((g - want).abs() - ulp).max())


def _fwd_bwd(march, leaves, grads_out, retain=False):
    lv = [None if x is None else x.detach().clone().requires_grad_(True) for x in leaves]
    out = march(*lv)
    outs = out if isinstance(out, tuple) else (out,)
    torch.autograd.backward(list(outs), list(grads_out), retain_graph=retain)
    torch.cuda.synchronize()
    return [o.detach() for o in outs], [None if x is None else x.grad for x in lv], (outs, lv)


def _assert_bf16_run_matches(march, s, grads_out, bf16_prims=False):
    """march(primpos, primrot, primscale, template, warp) with a bf16 template (and optionally bf16 primitive transforms) against
    the same call with their fp32 values."""
    t16 = s["template"].to(BF16)
    p16 = [s[k].to(BF16) if bf16_prims else s[k] for k in PRIMS]
    warp = s.get("warp")
    o32, g32, _ = _fwd_bwd(march, [p.float() for p in p16] + [t16.float(), warp], grads_out)
    o16, g16, _ = _fwd_bwd(march, p16 + [t16, warp], grads_out)
    for a, b in zip(o16, o32):
        assert a.dtype == torch.float32 and torch.equal(a, b)
    alpha16, alpha32 = (o16[0][..., 3], o32[0][..., 3]) if len(o16) == 1 else (o16[1], o32[1])
    assert float(alpha32.max()) > 0.0
    assert torch.equal(alpha16 >= 1.0, alpha32 >= 1.0)           # the same rays saturate
    _assert_within_bf16_ulp(g16[3], g32[3])
    for i in range(3):
        if bf16_prims:
            _assert_within_bf16_ulp(g16[i], g32[i])
        else:
            assert g16[i].dtype == torch.float32 and _trelerr(g16[i], g32[i]) <= ATOMIC_TOL, PRIMS[i]
    if warp is not None:
        assert g16[4].dtype == torch.float32 and _trelerr(g16[4], g32[4]) <= ATOMIC_TOL
    return o32


def _op(s, **kw):
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    algo = 1 if s.get("warp") is not None else 0
    fk = dict(fadescale=s.get("fadescale", 8.0), fadeexp=s.get("fadeexp", 8.0), algo=algo)
    fk.update(kw)
    return lambda pp, pr, ps, t, w: mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (pp, pr, ps), t, w, **fk)


def _cuda(s):
    return {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in s.items()}


@pytest.mark.parametrize("name", list(CASES))
def test_bf16_template_named_cases(name):
    s, grad = build_case(name)
    s = _cuda(s)
    _assert_bf16_run_matches(_op(s), s, [grad.cuda()])


def test_bf16_template_c2_full_size():
    """BASELINE.json config 2: 4 views 512x334, K=4096, 16^3."""
    s, grad = SAMPLED_CASES["c2"]()
    _assert_bf16_run_matches(_op(s), s, [grad])


def test_bf16_template_one_c3_view():
    """One full view of the benchmark scene (1024x667, K=16384, 8^3, alpha 17/6)."""
    from ava256_b200 import scene
    s = scene.make_scene(1, 1024, 667, 16384, 8, view_offset=5, alpha_mu=17.0, alpha_sigma=6.0, device="cuda")
    grad = torch.randn(1, 1024, 667, 4, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    out = _assert_bf16_run_matches(_op(s), s, [grad])
    assert float((out[0][..., 3] >= 1.0).float().mean()) > 0.005


def test_bf16_template_usebvh_true():
    s, grad = build_case("head_small")
    s = _cuda(s)
    _assert_bf16_run_matches(_op(s, usebvh=True), s, [grad.cuda()])


def test_bf16_template_shared_primitives():
    """[1,K,...] primitives and template rendered by all views (MVP_FLAG_SHARED_PRIMS)."""
    from ava256_b200 import scene
    s = scene.make_scene(3, 128, 96, 1024, 8, alpha_mu=10.0, alpha_sigma=5.0, device="cuda")
    for k in PRIMS + ("template",):
        s[k] = s[k][:1].contiguous()
    grad = torch.randn(3, 128, 96, 4, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    _assert_bf16_run_matches(_op(s), s, [grad])


@pytest.mark.parametrize("planes", [False, True])
def test_bf16_template_camera_entry_point(planes):
    from ava256_b200 import scene
    from ava256_b200.op import mvpraymarch_camera
    n, H, W = 2, 96, 70
    cams = [c.cuda() for c in scene.make_cameras(n, H, W, view_offset=2)]
    s = scene.make_scene(n, H, W, 256, 8, view_offset=2, alpha_mu=6.0, alpha_sigma=6.0, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(3)
    if planes:
        grads = [torch.randn(n, 3, H, W, device="cuda", generator=g), torch.randn(n, 1, H, W, device="cuda", generator=g)]
    else:
        grads = [torch.randn(n, H, W, 4, device="cuda", generator=g)]
    march = lambda pp, pr, ps, t, w: mvpraymarch_camera(*cams, (W, H), scene.VOLRADIUS, 1.0 / 64, (pp, pr, ps), t, w,  # noqa: E731
                                                       planes=planes)
    _assert_bf16_run_matches(march, s, grads)


def test_bf16_template_nograd_forward():
    s, _ = build_case("head_small")
    s = _cuda(s)
    march = _op(s)
    prims = [s[k] for k in PRIMS]
    t16 = s["template"].to(BF16)
    with torch.no_grad():
        a = march(*prims, t16, None)
        b = march(*prims, t16.float(), None)
    assert float(a[..., 3].max()) > 0.0 and torch.equal(a, b)


def test_bf16_template_second_backward():
    """retain_graph: the second backward gets new gradient buffers that the library zero-fills (MVP_FLAG_ZERO_GRADS)."""
    s, grad = build_case("head_small")
    s = _cuda(s)
    g = grad.cuda()
    t16 = s["template"].to(BF16)
    _, first, (outs, lv) = _fwd_bwd(_op(s), [s[k] for k in PRIMS] + [t16, None], [g], retain=True)
    first = [x.clone() for x in first[:4]]
    for x in lv[:4]:
        x.grad = None
    torch.autograd.backward(list(outs), [g])
    torch.cuda.synchronize()
    assert lv[3].grad.dtype == BF16
    for a, x in zip(first, lv[:4]):
        assert _trelerr(x.grad, a) <= ATOMIC_TOL
    _, g32, _ = _fwd_bwd(_op(s), [s[k] for k in PRIMS] + [t16.float(), None], [g])
    _assert_within_bf16_ulp(lv[3].grad, g32[3])


def test_bf16_template_row_bucket_overflow_and_512_cap():
    """K = 2304 slabs on the optical axis: the row buckets overflow and every tile goes to the 512-entry kernels."""
    from ava256_b200 import scene
    s = scene.make_scene(1, 16, 24, 2304, 2, alpha_mu=0.05, alpha_sigma=0.02)
    s["primpos"] = (s["primpos"] * 0.02).contiguous()
    s["stepsize"] = 1.0 / 16
    grad = torch.randn(1, 16, 24, 4, generator=torch.Generator().manual_seed(5))
    s = _cuda(s)
    _assert_bf16_run_matches(_op(s), s, [grad.cuda()])


@pytest.mark.parametrize("offset_bytes", [2, 8])
def test_bf16_template_view_at_an_offset(offset_bytes):
    """A contiguous bf16 template that starts inside a larger buffer: 2 bytes in (not 8-byte aligned: the op re-homes it) or
    8 bytes in (8- but not 16-byte aligned: read in place)."""
    from ava256_b200 import scene
    s = scene.make_scene(1, 64, 48, 64, 8, alpha_mu=6.0, alpha_sigma=4.0, device="cuda")
    grad = torch.randn(1, 64, 48, 4, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    t16 = s["template"].to(BF16)
    buf = torch.empty(t16.numel() + offset_bytes // 2, dtype=BF16, device="cuda")
    view = buf[offset_bytes // 2:].view(t16.shape)
    view.copy_(t16)
    assert view.data_ptr() % 16 == offset_bytes and view.is_contiguous()
    march = _op(s)
    prims = [s[k] for k in PRIMS]
    o_ref, g_ref, _ = _fwd_bwd(march, prims + [t16, None], [grad])
    out = march(*prims, view, None)                          # the view itself, not a re-homed clone
    assert torch.equal(out, o_ref[0])
    o_v, g_v, _ = _fwd_bwd(march, prims + [view, None], [grad])
    assert torch.equal(o_v[0], o_ref[0])
    _assert_within_bf16_ulp(g_v[3], g_ref[3].float())


def test_bf16_primitive_transforms():
    """primpos / primrot / primscale in bf16 (what bmm / linear give under autocast): the result of passing their fp32 values,
    gradients in bf16."""
    s, grad = build_case("head_small")
    s = _cuda(s)
    _assert_bf16_run_matches(_op(s), s, [grad.cuda()], bf16_prims=True)


def test_float16_template_raises():
    s, _ = build_case("head_small")
    s = _cuda(s)
    with pytest.raises(RuntimeError, match="float32 or bfloat16"):
        _op(s)(*[s[k] for k in PRIMS], s["template"].half(), None)
    with pytest.raises(RuntimeError, match="warp must be float32"):
        w = torch.zeros(2, 64, 2, 2, 2, 3, device="cuda", dtype=BF16)
        _op(s, algo=1)(*[s[k] for k in PRIMS], s["template"].to(BF16), w)
