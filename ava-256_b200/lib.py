"""ctypes binding of the C-ABI in include/mvpraymarch_b200.h.  There is no fallback: if the CUDA library cannot be
built or loaded, importing this module raises."""
import ctypes
import os

from . import build as _build

c_f = ctypes.c_void_p  # device pointers travel as plain addresses


class Shape(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("N", "H", "W", "K", "TD", "TH", "TW")]


class Camera(ctypes.Structure):
    """struct mvp_camera: the arguments of the reference's compute_raydirs on the integer pixel grid; viewpos == NULL = absent."""
    _fields_ = [("viewpos", c_f), ("viewrot", c_f), ("focal", c_f), ("princpt", c_f), ("volradius", ctypes.c_float),
                ("reserved", ctypes.c_uint32)]


class ForwardArgs(ctypes.Structure):
    """struct mvp_forward_args; the constructor fills struct_size."""
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("shape", Shape),
        ("stepsize", ctypes.c_float), ("fadescale", ctypes.c_float), ("fadeexp", ctypes.c_float),
        ("flags", ctypes.c_uint32),
        ("raypos", c_f), ("raydir", c_f), ("tminmax", c_f),
        ("primpos", c_f), ("primrot", c_f), ("primscale", c_f),
        ("tplate", c_f),
        ("rayrgba", c_f), ("raysat", c_f), ("rayaux", c_f),
        ("workspace", c_f), ("workspace_bytes", ctypes.c_size_t),
        ("warp", c_f), ("WD", ctypes.c_int32), ("WH", ctypes.c_int32), ("WW", ctypes.c_int32), ("algo", ctypes.c_int32),
        ("rayrgb_nchw", c_f), ("rayalpha_nchw", c_f), ("order", c_f),
        ("clear_grad_primpos", c_f), ("clear_grad_primrot", c_f), ("clear_grad_primscale", c_f), ("clear_grad_tplate", c_f),
        ("clear_grad_warp", c_f),
        ("camera", Camera),
    ]


class BackwardArgs(ctypes.Structure):
    """struct mvp_backward_args; the constructor fills struct_size."""
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("shape", Shape),
        ("stepsize", ctypes.c_float), ("fadescale", ctypes.c_float), ("fadeexp", ctypes.c_float),
        ("flags", ctypes.c_uint32),
        ("raypos", c_f), ("raydir", c_f), ("tminmax", c_f),
        ("primpos", c_f), ("primrot", c_f), ("primscale", c_f),
        ("tplate", c_f),
        ("grad_rayrgba", c_f), ("raysat", c_f), ("rayaux", c_f),
        ("grad_primpos", c_f), ("grad_primrot", c_f), ("grad_primscale", c_f), ("grad_tplate", c_f),
        ("workspace", c_f), ("workspace_bytes", ctypes.c_size_t),
        ("warp", c_f), ("grad_warp", c_f), ("WD", ctypes.c_int32), ("WH", ctypes.c_int32), ("WW", ctypes.c_int32),
        ("algo", ctypes.c_int32),
        ("grad_rayrgb_nchw", c_f), ("grad_rayalpha_nchw", c_f), ("order", c_f),
        ("camera", Camera),
    ]


def _sized_init(cls):
    def __init__(self, *a, **kw):
        ctypes.Structure.__init__(self, *a, **kw)
        self.struct_size = ctypes.sizeof(cls)
    cls.__init__ = __init__


_sized_init(ForwardArgs)
_sized_init(BackwardArgs)

FLAG_ACCEL_VALID = 1
FLAG_ZERO_GRADS = 2
FLAG_SHARED_PRIMS = 4
FLAG_TPLATE_BF16 = 8
FLAG_TEST_TINY_LISTS = 0x100
ABI_VERSION = 8
# layout pins, equal to the static_asserts in csrc/mvp_kernels.cu (tests/test_abi.py compares)
SIZEOF = {"Shape": 28, "Camera": 40, "ForwardArgs": 272, "BackwardArgs": 272}

EXPORTS = ("mvp_abi_version", "mvp_supported_flags", "mvp_build_config", "mvp_error_string", "mvp_workspace_bytes", "mvp_build_accel", "mvp_build_accel_camera",
           "mvp_raymarch_forward",
           "mvp_raymarch_backward", "mvp_compute_raydirs", "mvp_forward_launch_count", "mvp_backward_launch_count",
           "mvp_composite_forward", "mvp_composite_backward", "mvp_assemble_payload_forward",
           "mvp_assemble_payload_backward", "mvp_debug_saved_tiles", "mvp_debug_tileclk_offset", "mvp_compute_morton",
           "mvp_expand_views", "mvp_sum_views")


def _load():
    path = _build.LIB
    if _build.needs_build():
        try:
            _build.build()         # serialised across processes by a file lock, installed atomically (build.py)
        except Exception as e:
            # A prebuilt .so that travelled with the repo is acceptable only where it cannot be rebuilt (no nvcc on the
            # box); a failed compile of newer sources must not silently fall back to a stale library.
            if not os.path.exists(path) or _build.have_nvcc():
                raise RuntimeError("mvpraymarch_b200: CUDA library is missing or stale and could not be built: %r" % (e,))
            import warnings
            warnings.warn("mvpraymarch_b200: sources are newer than %s but nvcc is not available; loading the prebuilt library" % path)
    lib = ctypes.CDLL(path)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise RuntimeError("mvpraymarch_b200: %s does not export %s" % (path, name))
    lib.mvp_abi_version.restype = ctypes.c_int
    lib.mvp_supported_flags.restype = ctypes.c_int
    lib.mvp_supported_flags.argtypes = []
    lib.mvp_error_string.restype = ctypes.c_char_p
    lib.mvp_build_config.restype = ctypes.c_char_p
    lib.mvp_error_string.argtypes = [ctypes.c_int]
    lib.mvp_workspace_bytes.restype = ctypes.c_size_t
    lib.mvp_workspace_bytes.argtypes = [ctypes.POINTER(Shape)]
    lib.mvp_build_accel.restype = ctypes.c_int
    lib.mvp_build_accel.argtypes = [ctypes.POINTER(Shape), ctypes.c_uint32] + [c_f] * 7 + [ctypes.c_size_t, c_f]
    lib.mvp_build_accel_camera.restype = ctypes.c_int
    lib.mvp_build_accel_camera.argtypes = [ctypes.POINTER(Shape), ctypes.c_uint32, c_f, ctypes.POINTER(Camera)] + [c_f] * 4 + [ctypes.c_size_t, c_f]
    lib.mvp_compute_morton.restype = ctypes.c_int
    lib.mvp_compute_morton.argtypes = [ctypes.c_int32, ctypes.c_int32, c_f, c_f, c_f]
    lib.mvp_raymarch_forward.restype = ctypes.c_int
    lib.mvp_raymarch_forward.argtypes = [ctypes.POINTER(ForwardArgs), c_f]
    lib.mvp_raymarch_backward.restype = ctypes.c_int
    lib.mvp_raymarch_backward.argtypes = [ctypes.POINTER(BackwardArgs), c_f]
    lib.mvp_compute_raydirs.restype = ctypes.c_int
    lib.mvp_compute_raydirs.argtypes = [ctypes.c_int32] * 3 + [c_f] * 5 + [ctypes.c_float] + [c_f] * 4
    lib.mvp_composite_forward.restype = ctypes.c_int
    lib.mvp_composite_forward.argtypes = [ctypes.c_int32] * 3 + [c_f] * 7
    lib.mvp_composite_backward.restype = ctypes.c_int
    lib.mvp_composite_backward.argtypes = [ctypes.c_int32] * 3 + [c_f] * 10
    lib.mvp_expand_views.restype = ctypes.c_int
    lib.mvp_expand_views.argtypes = [c_f, c_f, ctypes.c_size_t, ctypes.c_int32, c_f]
    lib.mvp_sum_views.restype = ctypes.c_int
    lib.mvp_sum_views.argtypes = [c_f, c_f, ctypes.c_size_t, ctypes.c_int32, c_f]
    lib.mvp_assemble_payload_forward.restype = ctypes.c_int
    lib.mvp_assemble_payload_forward.argtypes = [ctypes.c_int32] * 4 + [c_f] * 2 + [ctypes.c_float] * 2 + [c_f] * 2
    lib.mvp_assemble_payload_backward.restype = ctypes.c_int
    lib.mvp_assemble_payload_backward.argtypes = [ctypes.c_int32] * 4 + [c_f] * 2 + [ctypes.c_float] + [c_f] * 3
    lib.mvp_forward_launch_count.restype = ctypes.c_int
    lib.mvp_forward_launch_count.argtypes = [ctypes.c_uint32]
    lib.mvp_backward_launch_count.restype = ctypes.c_int
    lib.mvp_backward_launch_count.argtypes = [ctypes.c_uint32]
    if lib.mvp_abi_version() != ABI_VERSION:
        raise RuntimeError("mvpraymarch_b200: ABI version mismatch (library %d, binding %d)" % (lib.mvp_abi_version(), ABI_VERSION))
    for cls in (Shape, Camera, ForwardArgs, BackwardArgs):
        assert ctypes.sizeof(cls) == SIZEOF[cls.__name__], cls.__name__
    return lib


LIB = _load()


def check(rc):
    if rc != 0:
        raise RuntimeError("mvpraymarch_b200: %s (code %d)" % (LIB.mvp_error_string(rc).decode(), rc))


def workspace_bytes(N, H, W, K, TD, TH, TW):
    s = Shape(N, H, W, K, TD, TH, TW)
    n = LIB.mvp_workspace_bytes(ctypes.byref(s))
    if n == 0:
        raise RuntimeError("mvpraymarch_b200: invalid shape %r" % ((N, H, W, K, TD, TH, TW),))
    return n
