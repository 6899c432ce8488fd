"""ctypes binding of `libsed_b200.so` (the C ABI declared in `include/sed_b200.h`).

There is no fallback: if the shared library is missing or an entry point fails, the caller gets an
exception.  torch is used only to obtain device pointers and the current CUDA stream.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsed_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "sed_b200.h")

SED_DTYPE_F16 = 0
SED_DTYPE_BF16 = 1
CONV_STORE, CONV_POOL, CONV_FREQMEAN = 0, 1, 2
LIVE_TABLE_COLS, LIVE_EVENT_STATE_INTS = 10, 19  # SED_LIVE_TABLE_COLS / SED_LIVE_EVENT_STATE_INTS
ERR_NAMES = {1: "SED_ERR_BAD_SHAPE", 2: "SED_ERR_UNSUPPORTED", 3: "SED_ERR_CUDA", 4: "SED_ERR_NULL",
             5: "SED_ERR_DRIVER"}

_p = ctypes.c_void_p
_i = ctypes.c_int
_l = ctypes.c_long
_f = ctypes.c_float
_d = ctypes.c_double

# name -> argtypes; mirrors include/sed_b200.h one to one (checked by tests/test_capi_symbols.py)
SIGNATURES = {
    "sed_abi_version": ([], _i),
    "sed_last_error_string": ([], ctypes.c_char_p),
    "sed_frontend_logmel": ([_p, _i, _i, _i, _l, _p, _l, _i, _i, _p, _p, _p, _p, _p, _p, _i, _f, _f, _i, _p, _p, _p, _p], _i),
    "sed_events": ([_p, _i, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p], _i),
    "sed_window_merge_avg": ([_p, _i, _i, _i, _i, _i, _i, _p, _p], _i),
    "sed_live_ingest": ([_p, _i, _p, _i, _l, _l, _p, _p], _i),
    "sed_live_merge": ([_p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p], _i),
    "sed_live_events": ([_p, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p], _i),
    "sed_resample_filter": ([_i, _i, _p, _p, _p, _p], _i),
    "sed_resample": ([_p, _i, _i, _p, _i, _l, _p, _i, _i, _i, _p, _p], _i),
    "sed_live_resample": ([_p, _i, _i, _p, _i, _l, _p, _i, _i, _i, _l, _p, _p, _i, _p, _i, _p], _i),
    "sed_spectrogram_f32": ([_p, _i, _i, _i, _i, _p, _p, _p, _p], _i),
    "sed_logmel_rows_f32": ([_p, _l, _i, _p, _p, _p, _p, _i, _f, _f, _i, _p, _p], _i),
    "sed_conv_first_f32": ([_p, _i, _i, _i, _p, _p, _p, _p, _i, _p], _i),
    "sed_conv3x3_bn_relu": ([_p, _i, _i, _i, _i, _p, _p, _p, _i, _i, _p, _p, _l, _l, _i, _p], _i),
    "sed_conv_block1": ([_p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _i, _p], _i),
    "sed_fold_bn": ([_p, _p, _p, _p, _i, _d, _p, _p, _p], _i),
    "sed_pack_conv3x3": ([_p, _i, _i, _p, _i, _p], _i),
    "sed_pack_conv_first": ([_p, _p, _p, _p], _i),
    "sed_pack_gru_whh": ([_p, _p, _p, _i, _p], _i),
    "sed_cast_16": ([_p, _l, _p, _i, _p], _i),
    "sed_count_saturated16": ([_p, _l, _i, _p, _p], _i),
    "sed_frontend_twiddle": ([_i, _p], _i),
    "sed_band_mel": ([_p, _i, _i, _p, _p, _p, _p, _i, _p], _i),
    "sed_fcpool": ([_p, _i, _i, _p, _p, _i, _i, _i, _p, _p, _p], _i),
    "sed_linear": ([_p, _l, _i, _p, _p, _i, _i, _p, _p, _i, _i, _p], _i),
    "sed_bigru_workspace_bytes": ([_i], _l),
    "sed_bigru": ([_p, _p, _p, _i, _i, _p, _p, _i, _p], _i),
    "sed_mha_core": ([_p, _i, _i, _l, _l, _p, _i, _p], _i),
    "sed_mha_attention": ([_p, _p, _i, _i, _l, _p, _i, _p], _i),
    "sed_linear_split16": ([_p, _l, _i, _p, _p, _i, _p, _p, _i, _i, _p], _i),
    "sed_attpool_blocks_scratch_bytes": ([_i, _i], _l),
    "sed_attpool_blocks": ([_p, _i, _i, _p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _i, _i, _i, _p], _i),
    "sed_peer_alloc": ([_l, _p], _i),
    "sed_peer_free": ([_p], _i),
    "sed_peer_export": ([_p, _p], _i),
    "sed_peer_open": ([_p, _p], _i),
    "sed_peer_close": ([_p], _i),
    "sed_peer_copy": ([_p, _p, _l, _p], _i),
    "sed_stream_write32": ([_p, ctypes.c_uint, _p], _i),
    "sed_stream_wait_geq32": ([_p, ctypes.c_uint, _p], _i),
    "sed_attpool": ([_p, _i, _i, _p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _p], _i),
}

_lib = None
_lock = threading.Lock()
_launches = 0  # kernels launched through this binding (reported by bench.py as gpu_launches)


class SedError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and type every entry point.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise SedError(
                "libsed_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C sound-event-detection_b200/csrc`. There is no CPU or PyTorch fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (argtypes, restype) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if a declared symbol is missing
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = lib
    return _lib


def use_profile_library():
    """Developer tools only: bind the -DSED_PROFILE build (`make -C csrc profile`), which carries the clock-stamp
    entry `sed_bigru_profile` and honours the SED_*_DBG experiment switches.  Must be called before load()."""
    global LIB_PATH
    if _lib is not None:
        raise SedError("use_profile_library() must be called before the library is loaded")
    LIB_PATH = os.path.join(_HERE, "libsed_b200_profile.so")
    SIGNATURES["sed_bigru_profile"] = ([_p, _p, _p, _i, _i, _p, _p, _i, _p, _p], _i)


def launches():
    return _launches


def reset_launches():
    global _launches
    _launches = 0


def _count(n=1):
    global _launches
    _launches += n


def check(rc, what):
    if rc != 0:
        msg = load().sed_last_error_string()
        msg = msg.decode("utf-8", "replace") if msg else ""
        exc = ValueError if rc in (1, 4) else NotImplementedError if rc == 2 else SedError
        raise exc("%s failed: %s (%s)" % (what, ERR_NAMES.get(rc, rc), msg))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def current_stream(device):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
