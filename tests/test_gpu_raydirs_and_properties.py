"""GPU tests: (1) ray generation (SURVEY 8f row 1) against the host formula and the reference's own kernel;
(2) the stand-alone accel / ACCEL_VALID C-ABI path; (3) size-independent properties at BASELINE.json's full
per-view sizes (C2: 512x334, K=4096, 16^3 and C3: 1024x667, K=16384, 8^3), where the CPU oracle is too slow."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.helpers import dome_cameras, relerr, sampled_relerr

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("with_pixelcoords", [False, True])
def test_compute_raydirs_matches_host_formula_and_reference(with_pixelcoords):
    """Against the host formula and against the reference's own kernel (its outputs stored as seeded samples,
    tests/golden/sampled_raydirs.npz)."""
    from ava256_b200 import scene
    from extensions.utils.utils import compute_raydirs
    n, H, W = 3, 77, 53
    campos, camrot, focal, princpt = dome_cameras(n, H, W)
    d = lambda t: t.cuda()  # noqa: E731
    if with_pixelcoords:
        py, px = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
        arg = torch.stack([px, py], dim=-1)[None].repeat(n, 1, 1, 1).contiguous().cuda()
    else:
        arg = (W, H)
    rp, rd, tmm = compute_raydirs(d(campos), d(camrot), d(focal), d(princpt), arg, scene.VOLRADIUS)
    hp, hd, ht = scene.compute_raydirs_host(campos, camrot, focal, princpt, H, W)
    assert relerr(rp.cpu().numpy(), hp.numpy()) < 1e-6
    assert relerr(rd.cpu().numpy(), hd.numpy()) < 1e-6
    assert relerr(tmm.cpu().numpy(), ht.numpy()) < 1e-5
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sampled_raydirs.npz"))
    tag = "pc1_" if with_pixelcoords else "pc0_"
    assert np.array_equal(rp.cpu().numpy(), gold[tag + "raypos"])
    assert sampled_relerr(rd, gold, tag + "raydir") < 2e-7
    assert sampled_relerr(tmm, gold, tag + "tminmax") < 1e-6


def test_generated_rays_render_like_host_rays():
    """Rays from our generator go down the pinhole fast path and give the oracle's image."""
    from ava256_b200 import scene
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    from extensions.utils.utils import compute_raydirs
    from oracle import oracle
    n, H, W, K, T = 1, 48, 32, 64, 8
    campos, camrot, focal, princpt = dome_cameras(n, H, W)
    rp, rd, tmm = compute_raydirs(campos.cuda(), camrot.cuda(), focal.cuda(), princpt.cuda(), (W, H), scene.VOLRADIUS)
    s = scene.make_scene(n, H, W, K, T, alpha_mu=2.0, alpha_sigma=2.0)
    with torch.no_grad():
        out = mvpraymarch(rp, rd, 1.0 / 32, tmm, (s["primpos"].cuda(), s["primrot"].cuda(), s["primscale"].cuda()),
                          s["template"].cuda(), None)
    ref, _ = oracle.forward(rp.cpu().numpy(), rd.cpu().numpy(), 1.0 / 32, tmm.cpu().numpy(), s["primpos"].numpy(),
                            s["primrot"].numpy(), s["primscale"].numpy(), s["template"].numpy())
    assert float(out[..., 3].max()) > 0.05
    assert relerr(out.cpu().numpy(), ref) <= 1e-4


def _abi_forward(s, flags, ws=None):
    from ava256_b200 import lib
    N, H, W = s["raypos"].shape[:3]
    K = s["primpos"].shape[1]
    T = s["template"].shape[2]
    P = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731
    wsb = lib.workspace_bytes(N, H, W, K, T, T, T)
    if ws is None:
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    rgba = torch.empty(N, H, W, 4, device="cuda")
    a = lib.ForwardArgs()
    a.shape = lib.Shape(N, H, W, K, T, T, T)
    a.stepsize, a.fadescale, a.fadeexp, a.flags = s["stepsize"], 8.0, 8.0, flags
    a.raypos, a.raydir, a.tminmax = P(s["raypos"]), P(s["raydir"]), P(s["tminmax"])
    a.primpos, a.primrot, a.primscale, a.tplate = P(s["primpos"]), P(s["primrot"]), P(s["primscale"]), P(s["template"])
    a.rayrgba, a.raysat, a.rayaux, a.workspace, a.workspace_bytes = P(rgba), None, None, P(ws), wsb
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(a), st))
    torch.cuda.synchronize()
    return rgba, ws


def test_standalone_accel_then_march_equals_one_shot():
    from ava256_b200 import lib, scene
    s = scene.make_scene(2, 96, 64, 256, 8, alpha_mu=4.0, alpha_sigma=3.0, device="cuda")
    one, _ = _abi_forward(s, 0)
    N, H, W = s["raypos"].shape[:3]
    wsb = lib.workspace_bytes(N, H, W, 256, 8, 8, 8)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    P = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731
    sh = lib.Shape(N, H, W, 256, 8, 8, 8)
    lib.check(lib.LIB.mvp_build_accel(ctypes.byref(sh), 0, None, P(s["raypos"]), P(s["raydir"]), P(s["primpos"]), P(s["primrot"]),
                                      P(s["primscale"]), P(ws), wsb, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    two, _ = _abi_forward(s, lib.FLAG_ACCEL_VALID, ws)
    assert torch.equal(one, two)


@pytest.mark.parametrize("cfg", [(2, 512, 334, 4096, 16), (1, 1024, 667, 16384, 8)], ids=["C2", "C3-view"])
def test_full_size_properties(cfg):
    """Determinism of forward, alpha range / saturation bookkeeping, linearity of backward in grad_rayrgba."""
    from ava256_b200 import scene
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    N, H, W, K, T = cfg
    s = scene.make_scene(N, H, W, K, T, alpha_mu=17.0, alpha_sigma=6.0, device="cuda")
    names = ("primpos", "primrot", "primscale", "template")

    def run(grad):
        lv = [s[n].clone().requires_grad_(True) for n in names]
        out = mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (lv[0], lv[1], lv[2]), lv[3], None)
        out.backward(grad)
        return out.detach(), [x.grad for x in lv]

    g = torch.randn(N, H, W, 4, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    o1, g1 = run(g)
    o2, g2 = run(2.0 * g)
    assert torch.equal(o1, o2), "forward must be deterministic"
    a = o1[..., 3]
    assert float(a.min()) >= 0.0 and float(a.max()) <= 1.0 + 1e-6
    cover = float((a > 0).float().mean())
    satur = float((a >= 1.0 - 1e-6).float().mean())
    assert 0.1 < cover < 0.6 and 0.02 < satur < cover
    assert bool(torch.isfinite(o1).all())
    for n_, x1, x2 in zip(names, g1, g2):
        assert bool(torch.isfinite(x1).all()), n_
        scale = float(x1.abs().max())
        assert scale > 0, n_
        # atomics reorder fp32 sums between runs: compare to 1e-4 of the tensor's scale
        assert float((x2 - 2.0 * x1).abs().max()) <= 1e-4 * 2.0 * scale, n_


def test_forward_is_cuda_graph_capturable():
    """No allocation, no sync, caller's stream inside the native call (INTEGRATION.md section 3): the whole forward,
    including the accel build and the programmatic-dependent-launch pair, can be captured and replayed."""
    from ava256_b200 import lib, scene
    s = scene.make_scene(1, 64, 48, 256, 8, alpha_mu=4.0, alpha_sigma=3.0, device="cuda")
    eager, _ = _abi_forward(s, 0)
    N, H, W = s["raypos"].shape[:3]
    P = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731
    wsb = lib.workspace_bytes(N, H, W, 256, 8, 8, 8)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    out = torch.zeros(N, H, W, 4, device="cuda")
    a = lib.ForwardArgs()
    a.shape = lib.Shape(N, H, W, 256, 8, 8, 8)
    a.stepsize, a.fadescale, a.fadeexp, a.flags = s["stepsize"], 8.0, 8.0, 0
    a.raypos, a.raydir, a.tminmax = P(s["raypos"]), P(s["raydir"]), P(s["tminmax"])
    a.primpos, a.primrot, a.primscale, a.tplate = P(s["primpos"]), P(s["primrot"]), P(s["primscale"]), P(s["template"])
    a.rayrgba, a.raysat, a.rayaux, a.workspace, a.workspace_bytes = P(out), None, None, P(ws), wsb
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(a), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.current_stream().wait_stream(side)
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
