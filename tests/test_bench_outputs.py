"""bench.py --dump-outputs: what the timed path computed in its last step, written as .npy files within 64 MB, the same
from run to run, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.helpers import relerr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUTPUTS = ("rayrgba", "grad_template", "grad_primpos", "grad_primrot", "grad_primscale")


def test_sample_outputs_keeps_small_arrays_whole_and_samples_rows_within_budget():
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = {"small": torch.randn(10, 3, generator=g), "big": torch.randn(5000, 4, generator=g),
              "bigger": torch.randn(20, 500, 4, generator=g)}
    a = bench.sample_outputs(arrays, budget=64_000)
    b = bench.sample_outputs(arrays, budget=64_000)
    assert sum(x.nbytes for x in a.values()) <= 64_000
    assert np.array_equal(a["small"], arrays["small"].numpy())
    for name in ("big", "bigger"):
        assert a[name].dtype == np.float32 and a[name].shape[1] == 4 and 1000 < a[name].shape[0] < 3000
        assert np.array_equal(a[name], b[name])
        rows = arrays[name].reshape(-1, 4).numpy()
        assert all((rows == r).all(axis=1).any() for r in a[name][:50])
    whole = bench.sample_outputs(arrays)
    for name, x in arrays.items():
        assert np.array_equal(whole[name], x.numpy())


def _bench(outdir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--views", "2",
           "--height", "96", "--width", "64", "--prims", "256", "--voxels", "8", "--no-e2e", "--no-cpu-baseline",
           "--no-shared-leg", "--no-check", "--dump-outputs", str(outdir)]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=str(outdir.parent), timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {n: np.load(outdir / (n + ".npy")) for n in OUTPUTS}


@pytest.mark.gpu
def test_dumped_outputs_are_those_of_the_op_and_repeat(tmp_path):
    """The dump equals the op's images and the view-summed gradients on bench.py's inputs, whatever the number of steps."""
    from ava256_b200 import scene
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    line1, a = _bench(tmp_path / "a", 1)
    line3, b = _bench(tmp_path / "b", 3)
    assert line1["steps"] == 1 and line3["steps"] == 3
    for n in OUTPUTS:
        assert a[n].dtype == np.float32
        assert relerr(a[n], b[n]) <= 1e-5, n
    assert np.array_equal(a["rayrgba"], b["rayrgba"])
    s = scene.make_scene(2, 96, 64, 256, 8, seed=1112, view_ids=[0, 1], device="cuda", alpha_mu=17.0, alpha_sigma=6.0)
    grad = torch.randn(2, 96, 64, 4, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1112))
    lv = [s[n].requires_grad_(True) for n in ("primpos", "primrot", "primscale", "template")]
    out = mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (lv[0], lv[1], lv[2]), lv[3], None)
    out.backward(grad)
    assert np.array_equal(a["rayrgba"], out.detach().cpu().numpy())
    for n, x in zip(("grad_primpos", "grad_primrot", "grad_primscale", "grad_template"), lv):
        assert a[n].shape == tuple(x.shape[1:])
        assert relerr(a[n], x.grad.sum(dim=0).cpu().numpy()) <= 1e-5, n
