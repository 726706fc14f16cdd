"""Shared test-input builders (seeded, CPU-generated so CPU and GPU runs see identical bytes)."""
import math

import numpy as np
import torch


def gradcheck_like_scene(N=2, H=13, W=13, k3=2, M=4, seed=1112, fadescale=6.5, fadeexp=7.5, alpha_gain=40.0, scale=2.2, dims=None):
    """Small scene in the style of the reference's gradcheck inputs
    (/root/reference/extensions/mvpraymarch/mvpraymarch.py:464-565): pinhole rays from z=-4, a k3^3 grid of
    randomly rotated slabs around the origin, softplus payload, random tminmax."""
    g = torch.Generator().manual_seed(seed)
    K = k3 ** 3
    focal = torch.tensor([[W * 4.0, W * 4.0]] * N)
    princpt = torch.tensor([[W * 0.5, H * 0.5]] * N)
    py, px = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
    pc = torch.stack([px, py], dim=-1)[None].repeat(N, 1, 1, 1)
    rd = (pc - princpt[:, None, None, :]) / focal[:, None, None, :]
    rd = torch.cat([rd, torch.ones_like(rd[..., :1])], dim=-1)
    rd = rd / rd.norm(dim=-1, keepdim=True)
    rp = torch.tensor([0.0, 0.0, -4.0])[None, None, None, :].repeat(N, H, W, 1)
    max_len = 6.0
    stepsize = max_len / 15.386928
    tminmax = max_len * torch.arange(2, dtype=torch.float32)[None, None, None, :].repeat(N, H, W, 1) \
        + torch.rand(N, H, W, 2, generator=g)
    TD, TH, TW = dims if dims is not None else (M, M, M)
    tpl = torch.nn.functional.softplus(1.5 * (torch.randn(N, K, TD, TH, TW, 4, generator=g)
                                              - torch.tensor([0, 0, 0, 3.5]))) * torch.tensor([1, 1, 1, alpha_gain])
    lin = torch.linspace(-1.0, 1.0, k3)
    gz, gy, gx = torch.meshgrid(lin, lin, lin, indexing="ij")
    grid = torch.stack([gx, gy, gz], dim=-1).reshape(1, K, 3)
    pos = 0.3 * (grid + 0.1 * torch.randn(N, K, 3, generator=g))
    rv = torch.randn(N * K, 3, generator=g)
    th = torch.sqrt(1e-5 + (rv ** 2).sum(-1, keepdim=True))
    kx = rv / th
    Kx = torch.zeros(N * K, 3, 3)
    Kx[:, 0, 1], Kx[:, 0, 2], Kx[:, 1, 0] = -kx[:, 2], kx[:, 1], kx[:, 2]
    Kx[:, 1, 2], Kx[:, 2, 0], Kx[:, 2, 1] = -kx[:, 0], -kx[:, 1], kx[:, 0]
    rot = (torch.eye(3)[None] + torch.sin(th)[..., None] * Kx + (1 - torch.cos(th))[..., None] * (Kx @ Kx)).view(N, K, 3, 3)
    scale = scale * torch.exp(0.1 * torch.randn(N, K, 3, generator=g))
    return dict(raypos=rp.contiguous(), raydir=rd.contiguous(), tminmax=tminmax.contiguous(), stepsize=stepsize,
                primpos=pos.contiguous(), primrot=rot.contiguous(), primscale=scale.contiguous(),
                template=tpl.contiguous(), fadescale=fadescale, fadeexp=fadeexp)


def make_warp(N, K, WD, WH, WW, seed=77, amp=0.05):
    """Warp field like the reference gradcheck's (mvpraymarch.py:498-510): identity grid + small noise; channels-last
    [N,K,WD,WH,WW,3] with channel order (x, y, z) = (W, H, D) axes."""
    g = torch.Generator().manual_seed(seed)
    lz, ly, lx = (torch.linspace(-1.0, 1.0, n) if n > 1 else torch.zeros(1) for n in (WD, WH, WW))
    gz, gy, gx = torch.meshgrid(lz, ly, lx, indexing="ij")
    grid = torch.stack([gx, gy, gz], dim=-1)[None, None]
    return (grid + amp * torch.randn(N, K, WD, WH, WW, 3, generator=g)).contiguous()


def scene_args_np(s, dtype=np.float32):
    """(positional args for oracle.forward, kwargs)."""
    a = [s["raypos"].numpy().astype(dtype), s["raydir"].numpy().astype(dtype), float(s["stepsize"]),
         s["tminmax"].numpy().astype(dtype), s["primpos"].numpy().astype(dtype), s["primrot"].numpy().astype(dtype),
         s["primscale"].numpy().astype(dtype), s["template"].numpy().astype(dtype)]
    kw = dict(fadescale=float(s.get("fadescale", 8.0)), fadeexp=float(s.get("fadeexp", 8.0)))
    if s.get("warp") is not None:
        kw["warp"] = s["warp"].numpy().astype(dtype)
    return a, kw


def relerr(a, b):
    """max|a-b| / max|b| -- the parity measure of SURVEY.md section 8d (the reference's own report format)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ----------------------------------------------------------------------------------------------------------
# Named, seeded parity cases (inputs are regenerated from seeds; tests/golden/*.npz hold reference OUTPUTS)
# ----------------------------------------------------------------------------------------------------------
def _head_case(n_views, H, W, K, T, seed=1112, view_offset=0, alpha_mu=6.0, alpha_sigma=6.0, stepsize=None):
    import sys, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    from ava256_b200 import scene
    s = scene.make_scene(n_views, H, W, K, T, seed=seed, view_offset=view_offset, alpha_mu=alpha_mu,
                         alpha_sigma=alpha_sigma, share_primitives=False)
    if stepsize is not None:
        s["stepsize"] = stepsize
    s["fadescale"], s["fadeexp"] = 8.0, 8.0
    return s


CASES = {
    # gradcheck-style (mvpraymarch.py:434-440 shapes scaled down), fade 6.5/7.5 like the reference's __main__ (:748-774)
    "gradcheck_small": lambda: gradcheck_like_scene(N=2, H=24, W=20, k3=3, M=6, seed=1112, alpha_gain=8.0),
    # odd image size (partial tiles in x and y), K not a power of two (rotated DFS order)
    "gradcheck_ragged": lambda: gradcheck_like_scene(N=1, H=13, W=19, k3=3, M=4, seed=7, alpha_gain=8.0),
    # head scene, C1-like but small: pinhole dome cameras, UV-grid slabs on an ellipsoid
    "head_small": lambda: _head_case(2, 64, 42, 64, 8, stepsize=1.0 / 64, alpha_mu=1.0, alpha_sigma=2.0),
    # 125 large overlapping slabs: every tile sees > 96 candidates -> exercises the 512-entry kernel variant
    "many_overlaps": lambda: gradcheck_like_scene(N=1, H=12, W=20, k3=5, M=4, seed=3, alpha_gain=0.4, scale=1.1),
    # non-cubic payload (runtime-stride sampler path) incl. a 1-voxel axis
    "noncubic": lambda: gradcheck_like_scene(N=1, H=14, W=17, k3=2, seed=21, alpha_gain=30.0, dims=(3, 1, 5)),
    # image smaller than one 8x4 tile, a single slab
    "tiny": lambda: gradcheck_like_scene(N=2, H=3, W=5, k3=1, M=2, seed=5, alpha_gain=15.0, scale=1.0),
    # algo 1: warp field (PrimSamplerTW<true>); large noise so warped positions leave the slab (zero padding)
    "warp_small": lambda: dict(gradcheck_like_scene(N=2, H=20, W=18, k3=2, M=6, seed=31, alpha_gain=60.0),
                               warp=make_warp(2, 8, 3, 4, 5, seed=5, amp=0.12)),
    "warp_head": lambda: dict(_head_case(1, 48, 32, 64, 8, stepsize=1.0 / 32, alpha_mu=2.0, alpha_sigma=2.0),
                              warp=make_warp(1, 64, 4, 4, 4, seed=9, amp=0.05)),
    # 18 views in one launch: above MVP_CTA_ORDER_MAXVIEWS (16), i.e. the large-launch forms of the accel build (warp-per-row
    # bucket kernel, plain grid order); every other case runs the small-launch forms
    "many_views": lambda: gradcheck_like_scene(N=18, H=9, W=11, k3=2, M=3, seed=13, alpha_gain=20.0),
    "head_t16": lambda: _head_case(1, 48, 32, 16, 16, stepsize=1.0 / 32, view_offset=11, alpha_mu=0.5, alpha_sigma=1.0),
}


def build_case(name):
    s = CASES[name]()
    g = torch.Generator().manual_seed(4242)
    grad = torch.randn(*s["raypos"].shape[:3], 4, generator=g)
    return s, grad


# ----------------------------------------------------------------------------------------------------------
# Scenes compared with the reference CUDA extension at sizes whose outputs are too large to store whole: a seeded sample
# of each reference output is kept in tests/golden/sampled_<name>.npz (tests/golden/make_sampled_golden.py)
# ----------------------------------------------------------------------------------------------------------
def _gpu_scene(n_views, H, W, K, T, alpha_mu, alpha_sigma, grad_seed, view_offset=0):
    from ava256_b200 import scene
    s = scene.make_scene(n_views, H, W, K, T, view_offset=view_offset, alpha_mu=alpha_mu, alpha_sigma=alpha_sigma, device="cuda")
    grad = torch.randn(n_views, H, W, 4, device="cuda", generator=torch.Generator(device="cuda").manual_seed(grad_seed))
    return s, grad


def _head_256x168():
    from ava256_b200 import scene
    s = scene.make_scene(2, 256, 168, 1024, 8, alpha_mu=3.0, alpha_sigma=3.0, share_primitives=False)
    return s, torch.randn(2, 256, 168, 4, generator=torch.Generator().manual_seed(99))


SAMPLED_CASES = {
    # BASELINE.json config 2: 1 subject, 4 views 512x334, K=4096, 16^3
    "c2": lambda: _gpu_scene(4, 512, 334, 4096, 16, 17.0, 6.0, 5),
    # the scene bench.py times (C3: 1024x667, K=16384, 8^3, alpha 17/6, dt=1/256), views 0, 1 and the two most oblique ones
    "c3_views0": lambda: _gpu_scene(2, 1024, 667, 16384, 8, 17.0, 6.0, 6, view_offset=0),
    "c3_views78": lambda: _gpu_scene(2, 1024, 667, 16384, 8, 17.0, 6.0, 84, view_offset=78),
    # mid-size head scene, inputs made on the CPU
    "head_256x168": _head_256x168,
}


def dome_cameras(n, H, W):
    """(campos, camrot, focal, princpt) of `n` dome cameras, fp32 on the CPU."""
    from ava256_b200 import scene
    campos, camrot = scene.look_at_cameras(n)
    ds = scene.FULLRES_H / H
    focal = torch.full((n, 2), scene.FOCAL_FULLRES / ds)
    princpt = torch.tensor([[W / 2.0, H / 2.0]]).expand(n, 2).contiguous()
    return campos.float().contiguous(), camrot.float().contiguous(), focal, princpt


def golden_sample(x, key, n=1024, seed=0):
    """Golden entries of tensor `x`: n element indices (half uniform over x, half uniform over its nonzero elements), the
    values there, and max|x| over the whole tensor."""
    flat = x.detach().reshape(-1)
    assert flat.numel() < 2 ** 31
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(flat.numel(), (n // 2,), generator=g)
    nz = flat.nonzero().view(-1).cpu()
    if nz.numel():
        idx = torch.cat([idx, nz[torch.randint(nz.numel(), (n - n // 2,), generator=g)]])
    idx = idx.unique()
    return {key + "__idx": idx.numpy().astype(np.int32), key + "__val": flat[idx.to(flat.device)].cpu().numpy(),
            key + "__absmax": np.float64(flat.abs().max().item())}


def sampled_relerr(x, gold, key):
    """relerr of tensor `x` against the reference tensor `key` of a golden_sample file, as far as the sample shows it: the
    larger of max|x - ref| over the sampled elements and |max|x| - max|ref||, over max|ref| of the whole tensor.  Both are
    lower bounds of max|x - ref| over the whole tensor, so any bound relerr(x, ref) meets holds for them too."""
    flat = x.detach().reshape(-1)
    idx = torch.from_numpy(gold[key + "__idx"].astype(np.int64)).to(flat.device)
    val = torch.from_numpy(gold[key + "__val"]).to(flat.device)
    absmax = float(gold[key + "__absmax"])
    d = float((flat[idx].double() - val.double()).abs().max())
    m = abs(float(flat.abs().max()) - absmax)
    return max(d, m) / max(absmax, 1e-30)


def golden_mask(mask, key):
    """A boolean tensor stored whole, one bit per element."""
    m = mask.detach().reshape(-1).cpu().numpy().astype(bool)
    return {key + "__bits": np.packbits(m), key + "__shape": np.array(mask.shape, np.int64)}


def load_golden_mask(gold, key):
    shape = tuple(int(v) for v in gold[key + "__shape"])
    return np.unpackbits(gold[key + "__bits"], count=int(np.prod(shape))).reshape(shape).astype(bool)


EDGE_KINDS = ("zero_scale", "rays_miss_volume", "large_step", "tiny_step")


def edge_scene(kind):
    s = gradcheck_like_scene(N=1, H=12, W=16, k3=2, M=4, seed=11, alpha_gain=30.0)
    if kind == "zero_scale":
        # SURVEY.md "input-distribution caveat": a decoder that skipped its warm-up feeds primscale = 0 (infinite slabs)
        s["primscale"][0, 1] = 0.0
        s["primscale"][0, 5, 2] = 0.0
    elif kind == "rays_miss_volume":
        # tmin > tmax for half of the rays (compute_raydirs gives that for rays missing the unit cube)
        s["tminmax"][0, :, :8, 0] = 9.0
        s["tminmax"][0, :, :8, 1] = 8.0
    elif kind == "large_step":
        s["stepsize"] = 1.7
    elif kind == "tiny_step":
        s["stepsize"] = 6.0 / 400.0
        s["template"][..., 3] *= 0.05
    return s
