"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Every call goes through the public op
(extensions.mvpraymarch.mvpraymarch.mvpraymarch -> ctypes -> C-ABI); the checkers are
  (a) oracle/mvp_oracle.c on the same seeded inputs,
  (b) the committed golden vectors produced by the unmodified reference CUDA extension (tests/golden/*.npz; at the
      mid-size head scene a seeded sample of them, tests/golden/sampled_*.npz).
Tolerances are the north star's: forward max|d|/max|ref| <= 1e-4, gradients <= 1e-3."""
import os

import numpy as np
import pytest
import torch

from tests.helpers import CASES, SAMPLED_CASES, build_case, edge_scene, relerr, sampled_relerr, scene_args_np

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-4
BWD_TOL = 1e-3
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def run_ours(s, grad=None):
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    dev = "cuda"
    t = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in s.items()}
    leaves = [t[k].clone().requires_grad_(grad is not None) for k in ("primpos", "primrot", "primscale", "template")]
    warp = t.get("warp")
    if warp is not None:
        warp = warp.clone().requires_grad_(grad is not None)
        leaves.append(warp)
    out = mvpraymarch(t["raypos"], t["raydir"], t["stepsize"], t["tminmax"], (leaves[0], leaves[1], leaves[2]), leaves[3],
                      warp, algo=1 if warp is not None else 0, fadescale=s.get("fadescale", 8.0), fadeexp=s.get("fadeexp", 8.0))
    if grad is None:
        return out.detach().cpu().numpy(), None
    out.backward(grad.to(dev))
    torch.cuda.synchronize()
    return out.detach().cpu().numpy(), [x.grad.cpu().numpy() for x in leaves]


@pytest.mark.parametrize("name", list(CASES))
def test_forward_backward_vs_oracle(name):
    from oracle import oracle
    s, grad = build_case(name)
    out, grads = run_ours(s, grad)
    a, kw = scene_args_np(s)
    ref, raysat = oracle.forward(*a, **kw)
    assert relerr(out, ref) <= FWD_TOL
    gref = oracle.backward(*a, grad.numpy(), raysat, **kw)
    assert len(grads) == len(gref)
    for nm, g, r in zip(("primpos", "primrot", "primscale", "template", "warp"), grads, gref):
        assert relerr(g, r) <= BWD_TOL, nm


@pytest.mark.parametrize("name", list(CASES))
def test_forward_backward_vs_golden(name):
    path = os.path.join(GOLDEN, name + ".npz")
    if not os.path.exists(path):
        pytest.skip("golden vector %s not generated yet" % name)
    gold = np.load(path)
    s, grad = build_case(name)
    out, grads = run_ours(s, grad)
    assert relerr(out, gold["rayrgba"]) <= FWD_TOL
    for nm, g in zip(("primpos", "primrot", "primscale", "template", "warp"), grads):
        assert relerr(g, gold["grad_" + nm]) <= BWD_TOL, nm


def test_nograd_forward_matches_grad_forward():
    s, _ = build_case("head_small")
    with torch.no_grad():
        a, _ = run_ours(s)
    b, _ = run_ours(s, torch.zeros(*s["raypos"].shape[:3], 4))
    assert np.array_equal(a, b)


def test_non_pinhole_rays_fall_back():
    """Rays that are not a pinhole grid (shuffled pixels) must still render correctly via the all-slabs fallback."""
    from oracle import oracle
    s, grad = build_case("gradcheck_ragged")
    g = torch.Generator().manual_seed(3)
    N, H, W = s["raypos"].shape[:3]
    perm = torch.randperm(H * W, generator=g)
    for k in ("raypos", "raydir", "tminmax"):
        v = s[k]
        s[k] = v.reshape(N, H * W, -1)[:, perm].reshape(v.shape).contiguous()
    out, grads = run_ours(s, grad)
    a, kw = scene_args_np(s)
    ref, raysat = oracle.forward(*a, **kw)
    assert relerr(out, ref) <= FWD_TOL
    gref = oracle.backward(*a, grad.numpy(), raysat, **kw)
    for nm, g_, r in zip(("primpos", "primrot", "primscale", "template"), grads, gref):
        assert relerr(g_, r) <= BWD_TOL, nm


def test_reference_extension_side_by_side():
    """Mid-size head scene against the reference kernels compiled for sm_100 (their outputs stored as seeded samples,
    tests/golden/sampled_head_256x168.npz)."""
    s, grad = SAMPLED_CASES["head_256x168"]()
    out, grads = run_ours(s, grad)
    gold = np.load(os.path.join(GOLDEN, "sampled_head_256x168.npz"))
    assert sampled_relerr(torch.from_numpy(out), gold, "rayrgba") <= FWD_TOL
    for nm, g_ in zip(("primpos", "primrot", "primscale", "template"), grads):
        assert sampled_relerr(torch.from_numpy(g_), gold, "grad_" + nm) <= BWD_TOL, nm


@pytest.mark.parametrize("kind", ["zero_scale", "rays_miss_volume", "large_step", "tiny_step"])
def test_edge_cases_vs_oracle(kind):
    from oracle import oracle
    s = edge_scene(kind)
    g = torch.Generator().manual_seed(17)
    grad = torch.randn(*s["raypos"].shape[:3], 4, generator=g)
    out, grads = run_ours(s, grad)
    a, kw = scene_args_np(s)
    ref, raysat = oracle.forward(*a, **kw)
    assert np.isfinite(out).all()
    assert relerr(out, ref) <= FWD_TOL
    gref = oracle.backward(*a, grad.numpy(), raysat, **kw)
    for nm, g_, r in zip(("primpos", "primrot", "primscale", "template"), grads, gref):
        assert np.isfinite(g_).all(), nm
        assert relerr(g_, r) <= BWD_TOL, nm


@pytest.mark.parametrize("name", ["head_small", "gradcheck_small", "warp_small"])
def test_usebvh_true_marches_in_morton_order(name):
    """usebvh=True == the fixed-order op on primitives gathered into Morton order (bit-exact), gradients scattered back;
    where nothing saturates the order is immaterial up to rounding."""
    from ava256_b200.op import morton_order
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    s, grad = build_case(name)
    t = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in s.items()}
    grad = grad.cuda()
    names = ["primpos", "primrot", "primscale", "template"] + (["warp"] if "warp" in t else [])
    kw = dict(algo=1 if "warp" in t else 0, fadescale=s.get("fadescale", 8.0), fadeexp=s.get("fadeexp", 8.0))

    def run(tensors, usebvh):
        leaves = {k: tensors[k].clone().requires_grad_(True) for k in names}
        out = mvpraymarch(t["raypos"], t["raydir"], t["stepsize"], t["tminmax"], (leaves["primpos"], leaves["primrot"], leaves["primscale"]),
                          leaves["template"], leaves.get("warp"), usebvh=usebvh, **kw)
        out.backward(grad)
        return out.detach(), {k: v.grad for k, v in leaves.items()}

    out_m, g_m = run(t, True)
    order = morton_order(t["primpos"])
    if name == "head_small":
        assert not torch.equal(order, torch.arange(order.size(1), device="cuda").expand_as(order))
    perm = {k: torch.gather(t[k], 1, order.view(order.shape + (1,) * (t[k].dim() - 2)).expand(order.shape + tuple(t[k].shape[2:]))).contiguous()
            for k in names}
    out_p, g_p = run(perm, "fixedorder")
    assert torch.equal(out_m, out_p)
    for k in names:
        back = torch.zeros_like(g_p[k]).scatter_(1, order.view(order.shape + (1,) * (g_p[k].dim() - 2)).expand_as(g_p[k]), g_p[k])
        assert relerr(g_m[k].cpu().numpy(), back.cpu().numpy()) < 1e-5, k
    out_f, _ = run(t, "fixedorder")
    unsat = (out_f[..., 3] < 0.999) & (out_m[..., 3] < 0.999)
    assert unsat.any()
    assert float((out_f - out_m)[unsat].abs().max()) <= 1e-4 * float(out_f.abs().max())


@pytest.mark.parametrize("seed", list(range(10)))
def test_random_small_scenes_vs_oracle(seed):
    """Seeded random shapes: image sizes that leave partial tiles, K that is not a power of two, cubic and non-cubic payloads,
    several views, step sizes from a handful to hundreds of steps per ray, with and without saturation -- against the oracle."""
    from oracle import oracle
    from tests.helpers import gradcheck_like_scene
    rng = np.random.default_rng(1000 + seed)
    N = int(rng.integers(1, 4))
    H, W = int(rng.integers(3, 30)), int(rng.integers(3, 40))
    k3 = int(rng.integers(1, 5))
    cubic = bool(rng.integers(0, 2))
    M = int(rng.choice([2, 3, 4, 8]))
    dims = None if cubic else (int(rng.integers(1, 6)), int(rng.integers(1, 6)), int(rng.integers(1, 6)))
    s = gradcheck_like_scene(N=N, H=H, W=W, k3=k3, M=M, seed=50 + seed, alpha_gain=float(rng.choice([0.5, 8.0, 60.0])),
                             scale=float(rng.uniform(0.9, 2.5)), dims=dims, fadescale=float(rng.uniform(4.0, 9.0)),
                             fadeexp=float(rng.uniform(5.0, 9.0)))
    s["stepsize"] = float(rng.choice([1.3, 0.39, 0.11, 0.03]))
    grad = torch.randn(N, H, W, 4, generator=torch.Generator().manual_seed(seed))
    out, grads = run_ours(s, grad)
    a, kw = scene_args_np(s)
    ref, raysat = oracle.forward(*a, **kw)
    assert np.isfinite(out).all() and relerr(out, ref) <= FWD_TOL
    gref = oracle.backward(*a, grad.numpy(), raysat, **kw)
    for nm, g_, r in zip(("primpos", "primrot", "primscale", "template"), grads, gref):
        assert np.isfinite(g_).all(), nm
        if np.abs(r).max() > 0:
            assert relerr(g_, r) <= BWD_TOL, nm


@pytest.mark.parametrize("name", ["head_small", "warp_small"])
def test_gradient_buffers_cleared_by_the_forward_and_second_backward(name):
    """The op hands the gradient buffers to the forward, whose render kernel zero-fills them (mvp_forward_args::clear_grad_*),
    and the backward runs without a memset pass; a second backward through the same graph (retain_graph) takes the library's
    zero-fill path instead.  Both give the same gradients, and they do not depend on what the allocator's blocks held before."""
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    s, grad = build_case(name)
    t = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in s.items()}
    junk = [torch.full((1 << 22,), float("nan"), device="cuda") for _ in range(4)]    # poison the allocator's free blocks
    del junk
    leaves = [t[k].clone().requires_grad_(True) for k in ("primpos", "primrot", "primscale", "template")]
    warp = t.get("warp")
    if warp is not None:
        warp = warp.clone().requires_grad_(True)
        leaves.append(warp)
    out = mvpraymarch(t["raypos"], t["raydir"], t["stepsize"], t["tminmax"], (leaves[0], leaves[1], leaves[2]), leaves[3], warp,
                      algo=1 if warp is not None else 0, fadescale=s.get("fadescale", 8.0), fadeexp=s.get("fadeexp", 8.0))
    g = grad.cuda()
    out.backward(g, retain_graph=True)
    first = [x.grad.clone() for x in leaves]
    for x in leaves:
        x.grad = None
    out.backward(g)
    _, ref = run_ours(s, grad)
    for a, b, c in zip(first, leaves, ref):
        assert torch.isfinite(a).all() and relerr(a.cpu().numpy(), c) <= 1e-5
        assert relerr(b.grad.cpu().numpy(), c) <= 1e-5
