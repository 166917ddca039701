"""ctypes binding of csrc/liblcpb200.so (the C ABI in include/lcpb200.h).

There is NO CPU fallback: importing the solver without the built library, or
calling it without a CUDA device, raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# LCPB200_LIB: load another build of the same library (debug / profiling builds); the default is the in-tree one
LIB_PATH = os.environ.get("LCPB200_LIB") or os.path.join(_HERE, "csrc", "liblcpb200.so")

F32, F64 = 0, 1
STATUS_SINGULAR_Q = -1

_lib = None

_vp = ctypes.c_void_p
_SIGS = {
    "lcpb200_version": (ctypes.c_int, []),
    "lcpb200_last_error_string": (ctypes.c_char_p, []),
    "lcpb200_create": (ctypes.c_int, [ctypes.c_int] * 5 + [ctypes.POINTER(_vp)]),
    "lcpb200_destroy": (ctypes.c_int, [_vp]),
    "lcpb200_workspace_bytes": (ctypes.c_size_t, [_vp]),
    "lcpb200_describe": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_size_t]),
    "lcpb200_profile": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.POINTER(ctypes.c_longlong)]),
    "lcpb200_forward": (ctypes.c_int, [_vp, ctypes.c_int] + [_vp] * 7 +
                        [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [_vp] * 9),
    "lcpb200_backward": (ctypes.c_int, [_vp, ctypes.c_int] + [_vp] * 17 + [ctypes.c_uint, _vp]),
    "lcpb200_forward_host": (ctypes.c_int, [_vp, ctypes.c_int] + [_vp] * 7 +
                             [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [_vp] * 7),
    "lcpb200_backward_host": (ctypes.c_int, [_vp, ctypes.c_int] + [_vp] * 16 + [ctypes.c_uint]),
    "lcpb200_engine_forward": (ctypes.c_int, [_vp] + [ctypes.c_int] * 4 + [ctypes.c_double] + [_vp] * 14 +
                               [ctypes.c_double, ctypes.c_int, ctypes.c_int] + [_vp] * 8),
    "lcpb200_engine_backward": (ctypes.c_int, [_vp] + [ctypes.c_int] * 4 + [ctypes.c_double] + [_vp] * 29 +
                                [ctypes.c_uint, _vp]),
    "lcpb200_find_contacts": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.c_double] + [_vp] * 6),
    "lcpb200_find_contacts_masked": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.c_double] + [_vp] * 7),
    "lcpb200_joint_rows": (ctypes.c_int, [ctypes.c_int] * 5 + [_vp] * 7),
    "lcpb200_joint_move": (ctypes.c_int, [ctypes.c_int] * 4 + [_vp] * 9),
    "lcpb200_contact_geometry": (ctypes.c_int, [ctypes.c_int] * 4 + [_vp] * 14),
    "lcpb200_assemble": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.c_double] + [_vp] * 17),
    "lcpb200_assemble_backward": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.c_double] + [_vp] * 25),
}
EXPORTS = tuple(_SIGS)


def load():
    """Load the shared library (once). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "lcp_physics_b200: CUDA library %s is missing. Build it with "
            "`python -m lcp_physics_b200.build` (needs nvcc). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("lcpb200: " + load().lcpb200_last_error_string().decode())


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("lcp_physics_b200 needs a CUDA device (B200, sm_100a); "
                           "there is no CPU fallback.")


def dtype_code(dtype):
    if dtype == torch.float32:
        return F32
    if dtype == torch.float64:
        return F64
    raise TypeError("lcp_physics_b200 supports float32 and float64, got %s" % dtype)


def ptr(t):
    """Raw data pointer of a tensor or None (NULL). Empty tensors map to NULL."""
    if t is None or t.numel() == 0:
        return None
    return ctypes.c_void_p(t.data_ptr())


class Handle:
    """Owns one lcpb200 handle (solver plan + workspace) for (dtype, n, m, e, device)."""

    def __init__(self, dtype, n, m, e, device_index):
        lib = load()
        self._h = _vp()
        check(lib.lcpb200_create(dtype_code(dtype), n, m, e, device_index, ctypes.byref(self._h)))
        self.key = (dtype, n, m, e, device_index)
        self.host_generation = 0        # bumped by every host-buffer call (retained-state token)
        self.fwd_generation = 0         # bumped by every device forward (structure-reuse token, lcp.py)

    def describe(self):
        buf = ctypes.create_string_buffer(512)
        check(load().lcpb200_describe(self._h, buf, 512))
        return buf.value.decode()

    def profile(self, enable=True):
        """Read (then reset or disable) the per-phase cycle counters: dict name -> SM cycles."""
        out = (ctypes.c_longlong * 24)()
        check(load().lcpb200_profile(self._h, 1 if enable else 0, out))
        return dict(zip(("prefactor", "load_T", "lu", "kkt_solve", "residual", "step", "lu_diag", "lu_panel",
                         "lu_update", "lu_inverse", "lu_slow_blocks", "lu_blocks", "lu_ahead", "lu_wait",
                         "c_structure", "c_block_inverse", "c_assemble", "c_lu", "c_solve_rhs", "c_solve_tri",
                         "c_solve_post", "c_residual", "c_step", "c_gradients"), list(out)))

    @property
    def raw(self):
        return self._h

    def __del__(self):
        try:
            if self._h:
                load().lcpb200_destroy(self._h)
                self._h = None
        except Exception:
            pass


_handles = {}          # insertion-ordered: least recently used first
_MAX_HANDLES = 32


def clear_handles():
    """Drop every cached handle (tests use it to re-plan under a different environment)."""
    _handles.clear()


def get_handle(dtype, n, m, e, device_index, stream=0):
    """One handle (plan + workspace) per (dtype, n, m, e, device, stream): the library's contract is one
    stream at a time per handle, so CUDA callers are keyed by their current stream and the host-buffer
    path (which runs on the handle's private streams) by stream = "host". LRU, at most 32 handles."""
    key = (dtype, n, m, e, device_index, stream)
    h = _handles.pop(key, None)
    if h is None:
        while len(_handles) >= _MAX_HANDLES:
            _handles.pop(next(iter(_handles)))
        h = Handle(dtype, n, m, e, device_index)
    _handles[key] = h
    return h
