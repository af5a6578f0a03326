"""ctypes binding of libucd_b200.so - the C ABI declared in include/ucd_b200.h.

This is the "reference-side FFI stub": the reference is pure PyTorch, so the maintainer-facing
binding is these ctypes prototypes plus the nn.Module classes in ucd_b200/losses.py.
There is no fallback: if the shared library is missing or fails to load, every entry point raises.
"""
import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libucd_b200.so")

_lib = None

UCD_ENOSUP = -3   # include/ucd_b200.h: a valid request this entry point does not take (the caller has another path)

P = c_void_p
_PROTOS = {
    "ucd_version": (c_int, []),
    "ucd_last_error": (ctypes.c_char_p, []),
    "ucd_device_ok": (c_int, []),
    "ucd_reduce_scratch_floats": (c_size_t, []),
    "ucd_unce_fwd": (c_int, [P, P, P, P, P, P, P, c_int, c_int, c_int, c_int64, c_int, P]),
    "ucd_unce_bwd": (c_int, [P, P, P, P, P, P, c_float, P, c_int, P, c_int, c_int, c_int, c_int, c_int64, c_int, P]),
    "ucd_unkd_fwd": (c_int, [P, P, P, c_float, P, P, P, P, c_int, c_int, c_int, c_int64, P]),
    "ucd_unkd_bwd": (c_int, [P, P, P, c_float, P, P, P, c_float, P, c_int, c_int, c_int, c_int, c_int64, P]),
    "ucd_kd_fwd": (c_int, [P, P, P, c_float, P, P, P, P, c_int, c_int, c_int, c_int64, c_int, c_float, P]),
    "ucd_kd_bwd": (c_int, [P, P, P, c_float, P, P, P, c_float, P, c_int, c_int, c_int, c_int, c_int64, c_int, P]),
    "ucd_unce_unkd_bwd": (c_int, [P, P, P, P, P, P, c_float, P, c_int, c_int, c_int, P, P, c_float, P, P, P, c_float, c_int,
                                  P, c_int, c_int, c_int, c_int, c_int64, P]),
    "ucd_unce_unkd_bwd_lowres": (c_int, [P, P, P, P, P, P, c_float, P, c_int, c_int, c_int, P, P, c_float, P, P, P,
                                         c_float, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ucd_bkg_mask": (c_int, [P, P, P, c_int, c_int, c_int64, c_int, P]),
    "ucd_upsample_bilinear_fwd": (c_int, [P, P, c_int64, c_int, c_int, c_int, c_int, P]),
    "ucd_upsample_bilinear_bwd": (c_int, [P, P, c_int64, c_int, c_int, c_int, c_int, P]),
    "ucd_upsample_argmax": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ucd_seg_fused_workspace_floats": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "ucd_seg_fused_fwd": (c_int, [P, P, P, P, P, P, P, c_size_t, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_int, c_int, c_float, c_int, P]),
    "ucd_con_max_tiles": (c_int64, [c_int64]),
    "ucd_con_prob_kpad": (c_int, [c_int]),
    "ucd_con_num_bins": (c_int, [c_int, c_int]),
    "ucd_con_px_meta_ints": (c_int64, [c_int64]),
    "ucd_con_blk_meta_ints": (c_int64, [c_int64, c_int]),
    "ucd_con_prep_labels": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P]),
    "ucd_con_prep_pack": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P, c_int, P, P, P, P,
                                  P, P, P, c_int64, P]),
    "ucd_con_prep_bwd": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int, P]),
    "ucd_con_prep_pack_bf16": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P, c_int, P, P, P,
                                       P, P, P, P, c_int64, P]),
    "ucd_con_prep_bwd_bf16": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int, P]),
    "ucd_rows_normalize_fwd": (c_int, [P, P, P, c_int, c_int, c_int, P]),
    "ucd_rows_normalize_bwd": (c_int, [P, P, P, P, c_int, c_int, c_int, P]),
    "ucd_con_tile_ranges": (c_int, [P, c_int64, P, P, P]),
    "ucd_con_pack_rows": (c_int, [P, P, c_int64, P, P, c_int64, P]),
    "ucd_con_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64]),
    "ucd_con_fwd": (c_int, [P, P, P, P, c_int, c_int64, c_int64, c_int, c_int, P, P, P, P, P, P, c_int64, P, c_int, c_int,
                            P, c_int64, c_float, c_int, P, P, P, c_size_t, c_int64, c_int64, P]),
    "ucd_con_bwd": (c_int, [P, P, P, c_float, P, P, P, c_int64, P]),
    "ucd_con_contrast_grad_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "ucd_con_contrast_grad": (c_int, [P, P, P, c_int, c_int64, c_int64, P, P, P, P, P, c_int64, c_int, P, c_int64,
                                      c_float, P, P, c_size_t, c_int64, c_int64, P]),
    "ucd_selfcon_workspace_bytes": (c_size_t, [c_int64]),
    "ucd_selfcon_fwd": (c_int, [P, P, P, P, P, c_int64, c_int64, c_int, c_float, c_float, c_int, P, P, P, c_size_t, P]),
}
EXPORTED = tuple(_PROTOS)
# include/ucd_b200_debug.h: exported by libucd_b200_debug.so only (python -m ucd_b200.build --debug)
_DEBUG_PROTOS = {
    "ucd_con_debug_trace": (c_int, [P]),
    "ucd_con_debug_splits": (c_int, [c_int64, c_int64]),
    "ucd_selftest_umma": (c_int, [c_int, ctypes.POINTER(c_float)]),
    "ucd_selftest_mma_rate": (c_int, [c_int, c_int, ctypes.POINTER(c_float)]),
    "ucd_selftest_mma_mix": (c_int, [c_int] * 8 + [ctypes.POINTER(c_float)]),
    "ucd_selftest_pipe_rate": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_float)]),
    "ucd_selftest_read_probe": (c_int, [P, ctypes.c_longlong, c_int, c_int, c_int, c_int, ctypes.POINTER(c_float)]),
}
DEBUG_EXPORTED = tuple(_DEBUG_PROTOS)
DEBUG_LIB_PATH = os.path.join(_HERE, "libucd_b200_debug.so")
_debug = None


def lib():
    """The loaded library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "ucd_b200: %s is missing - build it with `python -m ucd_b200.build` "
                "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)
        h = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def debug_lib(as_product=False):
    """The debug build (tracing, tuning knobs, tcgen05 probes); never used by the product modules.  With
    ``as_product=True`` the modules of this process run on it too (scripts that trace the product kernels)."""
    global _debug, _lib
    if _debug is None:
        if not os.path.exists(DEBUG_LIB_PATH):
            raise RuntimeError("ucd_b200: %s is missing - build it with `python -m ucd_b200.build --debug`" % DEBUG_LIB_PATH)
        h = ctypes.CDLL(DEBUG_LIB_PATH)
        for name, (res, args) in list(_PROTOS.items()) + list(_DEBUG_PROTOS.items()):
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _debug = h
    if as_product:
        _lib = _debug
    return _debug


class _NvtxProxy:
    """Wraps every kernel-launching C-ABI call in an NVTX range named after the entry point (SURVEY section 5:
    tracing), so that `ncu --nvtx --nvtx-include "ucd_con_fwd/"` (or nsys) can select the kernels of one call."""

    def __init__(self, handle):
        self._h = handle

    def __getattr__(self, name):
        fn = getattr(self._h, name)
        if not name.startswith("ucd_") or name in ("ucd_last_error", "ucd_version", "ucd_device_ok"):
            return fn
        import torch

        def wrapped(*args):
            torch.cuda.nvtx.range_push(name)
            try:
                return fn(*args)
            finally:
                torch.cuda.nvtx.range_pop()
        return wrapped


def enable_nvtx(on=True):
    """Turn NVTX ranges around the C-ABI calls of this process on or off (off by default: ~1 us per call)."""
    global _lib
    h = lib()
    if on and not isinstance(h, _NvtxProxy):
        _lib = _NvtxProxy(h)
    elif not on and isinstance(h, _NvtxProxy):
        _lib = h._h


def check(rc, what=""):
    if rc != 0:
        msg = lib().ucd_last_error().decode("utf-8", "replace")
        raise RuntimeError("ucd_b200 %s failed (code %d): %s" % (what, rc, msg))


def ptr(t):
    """Device pointer of a tensor (None -> NULL); a plain int is taken as a device address (section of a buffer whose
    typed view was never materialised as a tensor)."""
    if t is None:
        return None
    return c_void_p(t) if isinstance(t, int) else c_void_p(t.data_ptr())


_raw_stream = None


def cur_stream():
    """cudaStream_t of torch's current stream on the current device.  Uses torch's raw-stream accessor when it exists:
    `torch.cuda.current_stream()` builds a Stream object through several Python layers and was ~20 % of the host time of
    a step at small batch (scripts/host_profile.py)."""
    global _raw_stream
    import torch
    if _raw_stream is None:
        get_raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
        get_dev = getattr(torch._C, "_cuda_getDevice", None)
        if get_raw is not None and get_dev is not None:
            _raw_stream = lambda: get_raw(get_dev())                      # noqa: E731
        else:
            _raw_stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    return c_void_p(_raw_stream())
