"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol include/*.h declares, validates
arguments before touching a device, and the Python entry point keeps the reference's exact signature."""
import ctypes
import inspect
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REFERENCE_PARAMS = (  # /root/reference/extensions/mvpraymarch/mvpraymarch.py:295-318
    ("raypos", inspect.Parameter.empty), ("raydir", inspect.Parameter.empty), ("stepsize", inspect.Parameter.empty),
    ("tminmax", inspect.Parameter.empty), ("primtransf", inspect.Parameter.empty), ("template", inspect.Parameter.empty),
    ("warp", inspect.Parameter.empty), ("rayterm", None), ("algo", 0), ("usebvh", "fixedorder"), ("sortprims", False),
    ("randomorder", False), ("maxhitboxes", 512), ("synchitboxes", True), ("chlast", True), ("fadescale", 8.0),
    ("fadeexp", 8.0), ("accum", 0), ("termthresh", 0.0), ("griddim", 3), ("blocksize", (8, 16)), ("bwdblocksize", (8, 16)),
)


def test_header_symbols_are_exported():
    from ava256_b200 import lib
    hdr = open(os.path.join(ROOT, "include", "mvpraymarch_b200.h")).read()
    names = re.findall(r"^\s*(?:int|size_t|const char \*)\s*\**\s*(mvp_\w+)\s*\(", hdr, flags=re.M)
    assert set(names) >= {"mvp_raymarch_forward", "mvp_raymarch_backward", "mvp_build_accel", "mvp_workspace_bytes"}
    for n in names:
        assert hasattr(lib.LIB, n), n
    assert sorted(names) == sorted(lib.EXPORTS)
    assert lib.LIB.mvp_abi_version() == 8
    cfg = lib.LIB.mvp_build_config().decode()
    assert "LIST_REUSE=" in cfg and "FASTCAP=" in cfg and "CPU_EMUL" not in cfg


def test_c_program_through_the_header_alone(tmp_path):
    """A plain C program (tests/cabi/abi_probe.c) compiled against include/mvpraymarch_b200.h only: dlopen, every symbol
    it needs, struct sizes, the workspace query and the argument-error paths, with no Python in between.  The sizes it
    prints must be the ones the ctypes mirror (ava-256_b200/lib.py) and INTEGRATION.md use."""
    import subprocess
    from ava256_b200 import lib
    from ava256_b200 import build as _build
    exe = str(tmp_path / "abi_probe")
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cabi", "abi_probe.c"), "-o", exe, "-ldl"])
    out = subprocess.run([exe, _build.LIB], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    facts = dict(line.split(" ", 1) for line in out.stdout.strip().splitlines())
    assert facts["ok"] == "1" and int(facts["abi"]) == lib.ABI_VERSION
    assert int(facts["sizeof_shape"]) == ctypes.sizeof(lib.Shape) == lib.SIZEOF["Shape"]
    assert int(facts["sizeof_forward_args"]) == ctypes.sizeof(lib.ForwardArgs) == lib.SIZEOF["ForwardArgs"]
    assert int(facts["sizeof_backward_args"]) == ctypes.sizeof(lib.BackwardArgs) == lib.SIZEOF["BackwardArgs"]
    assert int(facts["sizeof_camera"]) == ctypes.sizeof(lib.Camera) == lib.SIZEOF["Camera"]
    assert int(facts["workspace_bytes_c3"]) == lib.workspace_bytes(80, 1024, 667, 16384, 8, 8, 8)
    # the stub printed in INTEGRATION.md states the same struct size
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert "ctypes.sizeof(ForwardArgs) == %d" % lib.SIZEOF["ForwardArgs"] in doc
    for field in ("struct_size", "workspace_bytes", '"warp"', '"WD"', '"WH"', '"WW"', '"algo"', '"rayrgb_nchw"', '"rayalpha_nchw"', '"order"', '"camera"'):
        assert field in doc, field


def test_truncated_argument_struct_is_rejected():
    from ava256_b200 import lib
    a = lib.ForwardArgs()
    assert a.struct_size == ctypes.sizeof(lib.ForwardArgs)
    a.struct_size -= 40                                                         # what an ABI-v7 caller (no `camera`) would pass
    assert lib.LIB.mvp_raymarch_forward(ctypes.byref(a), None) == -7          # MVP_ERR_STRUCT
    b = lib.BackwardArgs()
    b.struct_size = 0
    assert lib.LIB.mvp_raymarch_backward(ctypes.byref(b), None) == -7


def test_workspace_bytes_and_shape_validation():
    from ava256_b200 import lib
    small = lib.workspace_bytes(1, 128, 128, 256, 8, 8, 8)
    big = lib.workspace_bytes(80, 1024, 667, 16384, 8, 8, 8)
    assert 0 < small < big < 2 ** 31
    assert small % 256 == 0
    bad = lib.Shape(1, 0, 128, 256, 8, 8, 8)
    assert lib.LIB.mvp_workspace_bytes(ctypes.byref(bad)) == 0
    with pytest.raises(RuntimeError):
        lib.workspace_bytes(1, 40000, 128, 256, 8, 8, 8)


def test_argument_errors_do_not_need_a_device():
    from ava256_b200 import lib
    a = lib.ForwardArgs()
    a.shape = lib.Shape(1, 8, 8, 4, 2, 2, 2)
    a.stepsize = 0.1
    assert lib.LIB.mvp_raymarch_forward(ctypes.byref(a), None) == -1          # MVP_ERR_NULL
    assert lib.LIB.mvp_raymarch_forward(None, None) == -1
    dummy = ctypes.c_void_p(256)
    for f in ("raypos", "raydir", "tminmax", "primpos", "primrot", "primscale", "tplate", "rayrgba", "workspace"):
        setattr(a, f, dummy)
    a.workspace_bytes = 16
    assert lib.LIB.mvp_raymarch_forward(ctypes.byref(a), None) == -4          # MVP_ERR_WORKSPACE
    a.workspace_bytes = 1 << 30
    a.stepsize = 0.0
    assert lib.LIB.mvp_raymarch_forward(ctypes.byref(a), None) == -3          # MVP_ERR_STEPSIZE
    a.stepsize = float("nan")
    assert lib.LIB.mvp_raymarch_forward(ctypes.byref(a), None) == -3
    a.stepsize = 0.1
    a.shape = lib.Shape(1, 8, 8, 0, 2, 2, 2)
    assert lib.LIB.mvp_raymarch_forward(ctypes.byref(a), None) == -2          # MVP_ERR_SHAPE
    a.shape = lib.Shape(1, 8, 8, 4, 2, 2, 2)
    a.raysat = dummy                                                            # raysat without rayaux
    assert lib.LIB.mvp_raymarch_forward(ctypes.byref(a), None) == -1
    b = lib.BackwardArgs()
    assert lib.LIB.mvp_raymarch_backward(ctypes.byref(b), None) == -1
    assert b"workspace" in lib.LIB.mvp_error_string(-4)
    with pytest.raises(RuntimeError):
        lib.check(-2)


def test_python_entry_point_signature_matches_reference():
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    sig = inspect.signature(mvpraymarch)
    got = tuple((p.name, p.default) for p in sig.parameters.values())
    assert got == REFERENCE_PARAMS
    # models/raymarchers/mvpraymarcher.py:45 filters renderoptions with this attribute
    assert mvpraymarch.__code__.co_varnames[: len(REFERENCE_PARAMS)] == tuple(n for n, _ in REFERENCE_PARAMS)


def test_op_rejects_cpu_tensors_loudly():
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    from tests.helpers import build_case
    s, _ = build_case("gradcheck_ragged")
    with pytest.raises(RuntimeError, match="CUDA"):
        mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (s["primpos"], s["primrot"], s["primscale"]),
                    s["template"], None)


def test_camera_entry_point_has_no_cpu_path_either():
    """mvpraymarch_camera (compute_raydirs + mvpraymarch as one call): host tensors raise like the reference's CHECK_CUDA /
    AT_ASSERTM, for the fused form ((W, H) pixel grid) and for the two-call form (pixelcoords tensor) alike; the parameter list
    starts with compute_raydirs' own (extensions/utils/utils.py:48-51)."""
    from ava256_b200 import scene
    from ava256_b200.op import mvpraymarch_camera
    from tests.helpers import build_case
    s, _ = build_case("gradcheck_ragged")
    H, W = s["raypos"].shape[1:3]
    cams = scene.make_cameras(1, H, W)
    prim = (s["primpos"], s["primrot"], s["primscale"])
    assert list(inspect.signature(mvpraymarch_camera).parameters)[:6] == ["viewpos", "viewrot", "focal", "princpt", "pixelcoords", "volradius"]
    with pytest.raises(RuntimeError, match="CUDA"):
        mvpraymarch_camera(*cams, (W, H), 256.0, s["stepsize"], prim, s["template"], None)
    with pytest.raises(RuntimeError, match="CUDA"):
        mvpraymarch_camera(*cams, torch.zeros(1, H, W, 2), 256.0, s["stepsize"], prim, s["template"], None)


def test_unsupported_modes_raise():
    from extensions.mvpraymarch.mvpraymarch import mvpraymarch
    from tests.helpers import build_case
    s, _ = build_case("gradcheck_ragged")
    with pytest.raises(RuntimeError, match="warp"):
        mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (s["primpos"], s["primrot"], s["primscale"]),
                    s["template"], None, algo=1)
    with pytest.raises(NotImplementedError):
        mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (s["primpos"], s["primrot"], s["primscale"]),
                    s["template"], None, algo=2)
    with pytest.raises(NotImplementedError):
        mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (s["primpos"], s["primrot"], s["primscale"]),
                    s["template"], None, usebvh=False)
    with pytest.raises(RuntimeError, match="CUDA"):     # Morton mode is host logic + the same op: no CPU fallback either
        mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], (s["primpos"], s["primrot"], s["primscale"]),
                    s["template"], None, usebvh=True)


def test_morton_order_matches_bit_interleave():
    """usebvh=True order: op.morton_codes (the reference's magic-multiply expand_bits, bvh.cu:20-41) against a plain
    bit-by-bit interleave of the quantised centres, ties stable."""
    import numpy as np
    from ava256_b200.op import _take, morton_codes, morton_order
    g = torch.Generator().manual_seed(3)
    p = torch.rand(3, 97, 3, generator=g) * 2 - 1
    p[1, 5] = p[1, 50]                                   # a tie
    p[2, :, 2] = 0.25                                    # degenerate axis: (cmax - cmin) clamps to 1e-8 -> code bits 0
    c = morton_codes(p).numpy()
    cmax, cmin = p.max(1, keepdim=True)[0], p.min(1, keepdim=True)[0]
    q = ((p - cmin) / (cmax - cmin).clamp(min=1e-8) * 1024.0).clamp(0.0, 1023.0).to(torch.int64).numpy()
    ref = np.zeros(q.shape[:2], np.int64)
    for i in range(10):
        ref |= ((q[..., 0] >> i) & 1) << (3 * i + 2)
        ref |= ((q[..., 1] >> i) & 1) << (3 * i + 1)
        ref |= ((q[..., 2] >> i) & 1) << (3 * i)
    assert np.array_equal(c, ref) and c.max() < 2 ** 30 and c.min() >= 0
    o = morton_order(p).numpy()
    for n in range(3):
        assert sorted(o[n]) == list(range(97))
        cs = c[n][o[n]]
        assert (np.diff(cs) >= 0).all()
        same = np.diff(cs) == 0
        assert (np.diff(o[n])[same] > 0).all()           # stable
    assert list(o[1]).index(5) + 1 == list(o[1]).index(50)
    t = torch.rand(3, 97, 2, 3, generator=g, requires_grad=True)
    got = _take(t, torch.from_numpy(o))
    assert torch.equal(got[2, 7], t[2, o[2, 7]])
    got.backward(torch.ones_like(got))
    assert torch.equal(t.grad, torch.ones_like(t))


def test_scene_generator_is_deterministic_and_pinhole():
    from ava256_b200 import scene
    a = scene.make_scene(2, 32, 20, 16, 4)
    b = scene.make_scene(2, 32, 20, 16, 4)
    for k in a:
        if torch.is_tensor(a[k]):
            assert torch.equal(a[k], b[k]), k
    assert torch.allclose(a["raydir"].norm(dim=-1), torch.ones(2, 32, 20), atol=1e-5)
    assert (a["raypos"][0] == a["raypos"][0, 0, 0]).all()
    # rotations orthonormal, scales positive
    r = a["primrot"][0]
    assert torch.allclose(r @ r.transpose(1, 2), torch.eye(3).expand_as(r), atol=1e-4)
    assert (a["primscale"] > 0).all() and (a["template"] >= 0).all()


def test_overlay_resolves_from_unmodified_reference_modules(tmp_path):
    """With this repo in front of an ava-256 checkout, the checkout's modules import OUR op and ray generator
    (INTEGRATION.md section 1).  The checkout is a stand-in with the reference's package layout (no __init__.py under
    extensions/ or models/): its raymarcher module imports the op the way models/raymarchers/mvpraymarcher.py:14 does, and
    its own extension modules raise if they are ever imported."""
    import subprocess
    import sys
    ref = tmp_path / "ava-256"
    for rel in ("extensions/mvpraymarch/mvpraymarch.py", "extensions/utils/utils.py"):
        (ref / rel).parent.mkdir(parents=True)
        (ref / rel).write_text("raise ImportError('the checkout\\'s own %s was imported')\n" % rel)
    (ref / "models" / "raymarchers").mkdir(parents=True)
    (ref / "models" / "raymarchers" / "mvpraymarcher.py").write_text("from extensions.mvpraymarch.mvpraymarch import mvpraymarch\n")
    code = ("import models.raymarchers.mvpraymarcher as m, extensions.utils.utils as u, inspect;"
            "print(inspect.getsourcefile(m.mvpraymarch)); print(inspect.getsourcefile(u.compute_raydirs))")
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + str(ref))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = out.stdout.strip().splitlines()
    assert lines[0].startswith(ROOT) and "ava-256_b200" in lines[0]
    assert lines[1].startswith(ROOT) and "ava-256_b200" in lines[1]
