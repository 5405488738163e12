"""ctypes binding of libv100.so (C ABI in include/v100.h).

There is no fallback of any kind: if the shared library is missing or an entry point fails, the caller
gets an exception.  Build the library with `python -m voice100_b200.build`.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# V100_LIB selects an alternate build of the same ABI (same-box A/B measurements, tools/build_rev.sh)
LIB_PATH = os.path.abspath(os.environ["V100_LIB"]) if os.environ.get("V100_LIB") else os.path.join(_HERE, "libv100.so")

_p, _i, _l, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> argtypes; mirrors include/v100.h declaration by declaration
SIGNATURES = {
    "v100_abi_version": [],
    "v100_logmel": [_p, _i, _p, _i, _l, _i, _p, _p, _p, _p, _i, _f, _p, _i, _l, _i, _p, _p],
    "v100_logmel_generic": [_p, _i, _p, _i, _l, _i, _i, _i, _i, _i, _p, _p, _p, _p, _f, _p, _i, _l, _i, _p, _p],
    "v100_ntc_f32_to_ncw16": [_p, _p, _i, _i, _i, _l, _i, _p],
    "v100_ncw_f32_to_16": [_p, _p, _l, _i, _i, _i, _i, _p],
    "v100_ncw_16_to_f32": [_p, _l, _p, _i, _i, _i, _i, _p],
    "v100_conv1x1": [_p, _l, _p, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _i, _p],
    "v100_conv1x1_f32out": [_p, _l, _p, _p, _p, _l, _i, _i, _i, _i, _i, _p],
    "v100_dwconv1d": [_p, _l, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _i, _i, _p],
    "v100_dwconv1d_simt": [_p, _l, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _i, _i, _p],
    "v100_convtranspose1d_k5s2": [_p, _l, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _p],
    "v100_embedding_ncw16": [_p, _p, _p, _l, _i, _i, _i, _i, _p, _p],
    "v100_ctc_finalize": [_p, _l, _p, _p, _i, _i, _i, _p, _p, _p],
    "v100_ctc_collapse": [_p, _p, _p, _p, _i, _i, _i, _p],
    "v100_ctc_best_path": [_p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p],
    "v100_world_finalize": [_p, _l, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p],
    "v100_ncw_f32_to_ntc": [_p, _l, _p, _i, _i, _i, _p],
    "v100_maskaudio": [_p, _p, _p, _i, _i, _i, _f, _p],
    "v100_conv1d": [_p, _l, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _i, _i, _i, _p],
    "v100_conv1d_tm": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p],
    "v100_layernorm_gelu": [_p, _l, _p, _p, _f, _p, _l, _i, _i, _i, _i, _p],
    "v100_ncw_to_tm": [_p, _l, _p, _i, _i, _i, _i, _p],
    "v100_tm_to_ncw": [_p, _p, _l, _i, _i, _i, _i, _p],
    "v100_lstm_layer": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p],
    "v100_tts_align": [_p, _l, _l, _l, _i, _p, _p, _l, _p, _i, _i, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p],
    "v100_world_noise": [_p, _l, _p],
    "v100_world_workspace_bytes": [_i, _l],   # returns int64 (restype set in lib())
    "v100_world_timebase": [_p, _l, _l, _p, _l, _l, _l, _p, _l, _l, _p, _i, _i, _p, _p, _p, _p],
    "v100_world_synthesize": [_p, _l, _l, _p, _l, _l, _l, _p, _l, _l, _p, _i, _i, _p, _l, _p, _p, _l, _p, _p, _p],
    "v100_resample": [_p, _i, _p, _i, _l, _l, _p, _p, _p, _p, _i, _i, _i, _i, _p, _l, _l, _p, _p],
    "v100_world_analysis_workspace_bytes": [_i, _l],   # returns int64 (restype set in lib())
    "v100_world_analyze": [_p, _i, _l, _p, _i, _l, _p, _p, _l, _p, _i, _p, _p, _p, _p, _p, _p],
    "v100_ctc_loss": [_p, _l, _l, _i, _i, _i, _p, _p, _l, _p, _l, _p, _i, _i, _i, _i, _p, _p, _p],
    "v100_edit_distance": [_p, _l, _p, _i, _p, _l, _p, _i, _i, _p, _p],
}

ABI_VERSION = 9
_lib = None


class V100Error(RuntimeError):
    pass


def lib():
    """Load libv100.so once; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise V100Error(f"{LIB_PATH} is missing: run `python -m voice100_b200.build` (there is no CPU/PyTorch "
                            "fallback for the Voice100 hot path)")
        handle = C.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = _i
        handle.v100_lstm_workspace_bytes.argtypes = [_i, _i]
        handle.v100_lstm_workspace_bytes.restype = _l
        handle.v100_world_workspace_bytes.restype = _l
        handle.v100_world_analysis_workspace_bytes.restype = _l
        handle.v100_last_error.argtypes = []
        handle.v100_last_error.restype = C.c_char_p
        if handle.v100_abi_version() != ABI_VERSION:
            raise V100Error("libv100.so ABI version mismatch: rebuild with `python -m voice100_b200.build --force`")
        _lib = handle
    return _lib


# kernels launched per entry point (everything is one kernel except the transposed conv, which first
# builds its shifted channel stack)
KERNELS_PER_CALL = {name: 1 for name in SIGNATURES}
KERNELS_PER_CALL["v100_convtranspose1d_k5s2"] = 2
KERNELS_PER_CALL["v100_conv1d"] = 2   # tap stacking + GEMM
KERNELS_PER_CALL["v100_abi_version"] = 0
KERNELS_PER_CALL["v100_world_synthesize"] = 2   # time base + synthesis
KERNELS_PER_CALL["v100_world_workspace_bytes"] = 0
KERNELS_PER_CALL["v100_world_analysis_workspace_bytes"] = 0
KERNELS_PER_CALL["v100_world_analyze"] = 13     # prep, low-cut, bands x2, scan, contour, fix, StoneMask, draws x2,
                                                # CheapTrick, LoveTrain, D4C

stats = {"launches": 0}
tracer = None  # optional object with before(name)/after(name), used by bench.py for per-kernel CUDA events


def call(name, *args):
    """Invoke an entry point; non-zero status raises with the library's own message."""
    handle = lib()
    if tracer is not None:
        tracer.before(name)
    rc = getattr(handle, name)(*args)
    if tracer is not None:
        tracer.after(name)
    if rc != 0:
        raise V100Error(f"{name} failed (status {rc}): {handle.v100_last_error().decode()}")
    stats["launches"] += KERNELS_PER_CALL[name]
