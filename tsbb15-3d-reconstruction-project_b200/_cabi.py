"""ctypes binding of librg_b200.so (the C ABI declared in include/rg_b200.h).

There is deliberately no fallback: if the shared library is missing, or the machine has no sm_100 GPU, every
product entry point raises.  Build the library with ``python __graft_entry__.py`` (or ``build.py``).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RG_LIB", os.path.join(_HERE, "librg_b200.so"))   # RG_LIB: kernel-variant experiments

MODE_EPI_MAX, MODE_SAMPSON = 0, 1
TIE_FIRST, TIE_REFERENCE = 0, 1
SOLVER_QR, SOLVER_JACOBI = 0, 1
SCORE_FP32_GUARDED, SCORE_FP64, SCORE_FP32_BOUND = 0, 1, 2
TRI_OPTIMAL, TRI_LINEAR = 0, 1
FLAG_REUSE_POINTS = 1
FLAG_BOUNDED = 2
LOSS_LINEAR, LOSS_SOFT_L1, LOSS_HUBER, LOSS_CAUCHY, LOSS_ARCTAN = 0, 1, 2, 3, 4

_vp = C.c_void_p
_i = C.c_int
_d = C.c_double
_pd = C.POINTER(C.c_double)
_pll = C.POINTER(C.c_longlong)

# name -> (restype, argtypes); mirrors include/rg_b200.h one to one (tests check every symbol is exported).  Buffers,
# the int32 offset tables included, are declared void*: ``call`` passes numpy arrays, tensors and addresses through ``ptr``.
SIGNATURES = {
    "rg_abi_version": (_i, []),
    "rg_last_error": (C.c_char_p, []),
    "rg_init": (_i, [_i, C.POINTER(_vp)]),
    "rg_shutdown": (_i, [_vp]),
    "rg_device_sm_count": (_i, [_vp]),
    "rg_host_alloc": (_i, [C.c_size_t, C.POINTER(_vp)]),
    "rg_host_free": (_i, [_vp]),
    "rg_set_option": (_i, [_vp, _i, C.c_longlong]),
    "rg_get_profile": (_i, [_vp, _vp, _pd, C.POINTER(C.c_int)]),
    "rg_microbench_run": (_i, [_pd, _vp]),
    "rg_get_last_stats": (_i, [_vp, _vp, _pll]),
    "rg_f_ransac_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "rg_f_ransac_dev2": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _i, C.c_ulonglong, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "rg_f_ransac_host2": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, C.c_ulonglong, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rg_sample_indices_dev": (_i, [_vp, _vp, _i, _vp, _vp, _i, C.c_ulonglong, _i, _i, _vp]),
    "rg_synth_two_view_dev": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp, C.c_ulonglong, _d, _d, _d, _d, _vp, _vp]),
    "rg_f_inlier_mask_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _d, _i, _vp]),
    "rg_pnp_ransac_batched_dev2": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "rg_p2p_create": (_i, [_vp, _i, _i, _vp]),
    "rg_p2p_connect": (_i, [_vp, _vp]),
    "rg_p2p_destroy": (_i, [_vp]),
    "rg_p2p_argmax_exchange": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "rg_f_last_hypotheses_dev": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "rg_f_last_bounded_stats": (_i, [_vp, _vp, _pll]),
    "rg_f_last_bounded_evals": (_i, [_vp, _vp, _pll]),
    "rg_f_ransac_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rg_f8pt_solve_host": (_i, [_vp, _vp, _i, _vp, _i, _vp, _i, _vp, _vp]),
    "rg_epi_score_count_host": (_i, [_vp, _vp, _i, _vp, _i, _vp, _d, _i, _i, _vp]),
    "rg_fmatrix_residuals_host": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "rg_fmatrix_stls_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "rg_pnp_ransac_host": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _vp, _d, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rg_pnp_ransac_dev": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _vp, _d, _i, _vp, _vp, _vp, _vp]),
    "rg_pnp_ransac_batched_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rg_pnp_ransac_batched_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _i, _vp, _vp, _vp, _vp]),
    "rg_pnp_minimize_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "rg_pnp_score_count_host": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _d, _i, _vp]),
    "rg_triangulate_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "rg_triangulate_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "rg_fmatrix_from_cameras_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "rg_relative_pose_host": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "rg_relative_pose_dev": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "rg_camera_resectioning_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "rg_gold_standard_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    "rg_gold_standard_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    "rg_gold_standard_host2": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _d, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    "rg_gold_standard_dev2": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _d, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    "rg_pnp_refine_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _i, _d, _vp, _vp, _vp, _vp]),
    "rg_pnp_refine_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _i, _d, _vp, _vp, _vp, _vp]),
    "rg_pnp_refine_host2": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _i, _d, _i, _d, _vp, _vp, _vp, _vp]),
    "rg_pnp_refine_dev2": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _i, _d, _i, _d, _vp, _vp, _vp, _vp]),
    "rg_fmatrix_residuals_gs_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "rg_bundle_adjust_host": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _d, _vp, _vp, _vp]),
    "rg_bundle_adjust_dev": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _d, _vp, _vp, _vp]),
    "rg_bundle_adjust_host2": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _d, _i, _d, _vp, _vp, _vp]),
    "rg_bundle_adjust_dev2": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _d, _i, _d, _vp, _vp, _vp]),
    "rg_ba_residuals_host": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rg_two_view_init_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rg_two_view_init_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rg_match_first_within_host": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _d, _vp]),
    "rg_argmax_pack_dev": (_i, [_vp, _i, _vp, _vp, _i, _vp]),
    "rg_argmax_allreduce": (_i, [_vp, _vp, _vp, _i]),
    "rg_argmax_unpack_dev": (_i, [_vp, _i, _vp, _vp, _vp]),
    "rg_match_first_within_dev": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _d, _vp]),
}

_lib = None
_calls: dict = {}                 # name -> (function, one argument converter per argtype), filled by load_library
_lock = threading.Lock()
_contexts: dict[int, int] = {}


class RGError(RuntimeError):
    """A librg_b200 call failed (message from rg_last_error)."""


def load_library() -> C.CDLL:
    """dlopen the in-tree library and declare every prototype.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.isfile(LIB_PATH):
                raise RGError(
                    f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                    "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
                _calls[name] = (fn, [_CONVERT.get(a, _same) for a in args])
            _lib = lib
    return _lib


def call(name: str, *args) -> None:
    """Calls the library entry point ``name``; raises through ``check`` when it fails.  Each argument is converted for
    its declared C type: a pointer takes None (NULL), a numpy array, a torch tensor or an int address (see ``ptr``), a
    number takes a Python or numpy scalar, and any other type (ctypes out-parameters) is passed as given."""
    if _lib is None:                      # set only after every prototype is declared
        load_library()
    fn, conv = _calls[name]
    if len(args) != len(conv):
        raise TypeError(f"{name} takes {len(conv)} arguments ({len(args)} given)")
    check(fn(*[c(a) for c, a in zip(conv, args)]))


def check(rc: int) -> None:
    if rc != 0:
        msg = load_library().rg_last_error()
        text = msg.decode("utf-8", "replace") if msg else ""
        if rc == -2:
            raise ValueError(f"librg_b200: {text}")
        raise RGError(f"librg_b200 call failed (code {rc}): {text}")


def context(device: int | None = None) -> int:
    """Lazily created per-device context handle (an opaque pointer as int)."""
    lib = load_library()
    if device is None:
        device = int(os.environ.get("RG_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    with _lock:
        if device not in _contexts:
            h = _vp()
            check(lib.rg_init(int(device), C.byref(h)))
            _contexts[device] = h.value
        return _contexts[device]


def shutdown_all() -> None:
    lib = load_library()
    with _lock:
        for dev, h in list(_contexts.items()):
            lib.rg_shutdown(_vp(h))
            del _contexts[dev]


def pinned_empty(shape, dtype, device: int | None = None) -> np.ndarray:
    """An uninitialised array in page-locked host memory (rg_host_alloc), freed when the array is collected.  Falls back
    to ordinary memory when the library or a CUDA device is not usable (this only affects upload speed, never results)."""
    import weakref
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    try:
        lib = load_library()
        context(device)                             # a context on the TARGET device must exist before page-locking
        p = _vp()
        if lib.rg_host_alloc(n, C.byref(p)) != 0 or not p.value:
            raise RGError("rg_host_alloc failed")
    except (RGError, OSError):
        return np.empty(shape, dtype=dtype)
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    weakref.finalize(buf, lib.rg_host_free, _vp(p.value))
    return arr


def ptr(a) -> int | None:
    """Raw address of a numpy array / torch tensor / int / ctypes c_void_p; None stays NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if isinstance(a, (int, np.integer)):
        return int(a)
    if hasattr(a, "data_ptr"):
        return int(a.data_ptr())
    if isinstance(a, C.c_void_p):
        return a.value
    raise TypeError(f"cannot take the address of {type(a)!r}")


def _same(a):
    return a


_CONVERT = {_vp: ptr, _d: float, _i: int, C.c_longlong: int, C.c_ulonglong: int, C.c_size_t: int}
