"""Generates tests/golden/sampled_*.npz on a GPU from the unmodified reference CUDA extension (oracle/_ref, built by
oracle/build_ref.py).  Its outputs for the scenes of tests/helpers.py SAMPLED_CASES and for the ray generator test are
hundreds of MB, so each output is stored as a seeded sample (tests/helpers.py golden_sample); the saturated-ray masks are
stored whole, one bit per ray.

    python tests/golden/make_sampled_golden.py OUTDIR [case ...]      # then copy OUTDIR/*.npz here
"""
import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import refext  # noqa: E402
from tests.helpers import SAMPLED_CASES, dome_cameras, golden_mask, golden_sample  # noqa: E402

NAMES = ("primpos", "primrot", "primscale", "template")


def _sample(x, key):
    return golden_sample(x, key, seed=zlib.crc32(key.encode()))


def raymarch_case(name):
    s, grad = SAMPLED_CASES[name]()
    t = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in s.items()}
    rgba, sat, st = refext.forward(t["raypos"], t["raydir"], t["stepsize"], t["tminmax"], t["primpos"], t["primrot"],
                                   t["primscale"], t["template"])
    g = refext.backward(t["raypos"], t["raydir"], t["stepsize"], t["tminmax"], t["primpos"], t["primrot"], t["primscale"],
                        t["template"], rgba, sat, st, grad.cuda())
    out = dict(_sample(rgba, "rayrgba"), **golden_mask(sat[..., 0] > -1.0, "saturated"))
    for nm, x in zip(NAMES, g):
        out.update(_sample(x, "grad_" + nm))
    return out


def raydirs_case(n=3, H=77, W=53):
    """compute_raydirs of the reference, with the integer pixel grid given as (W, H) ("pc0_") and as a tensor ("pc1_")."""
    from ava256_b200 import scene
    cams = [c.cuda() for c in dome_cameras(n, H, W)]
    py, px = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
    pc = torch.stack([px, py], dim=-1)[None].repeat(n, 1, 1, 1).contiguous().cuda()
    out = {}
    for tag, p in (("pc0_", None), ("pc1_", pc)):
        rp, rd, tmm = refext.compute_raydirs(*cams, p, H, W, scene.VOLRADIUS)
        out[tag + "raypos"] = rp.cpu().numpy()
        out.update(_sample(rd, tag + "raydir"))
        out.update(_sample(tmm, tag + "tminmax"))
    return out


def main(outdir, only=()):
    os.makedirs(outdir, exist_ok=True)
    jobs = [(n, lambda n=n: raymarch_case(n)) for n in SAMPLED_CASES] + [("raydirs", raydirs_case)]
    for name, fn in jobs:
        if only and name not in only:
            continue
        path = os.path.join(outdir, "sampled_%s.npz" % name)
        np.savez_compressed(path, **fn())
        torch.cuda.empty_cache()
        print(name, "saved:", os.path.getsize(path), "bytes", flush=True)


if __name__ == "__main__":
    main(sys.argv[1], tuple(sys.argv[2:]))
