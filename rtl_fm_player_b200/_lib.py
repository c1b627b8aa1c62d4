"""ctypes binding of the C ABI in include/fmb.h (rtl_fm_player_b200/libfmb.so).

The shared library is the product; this module only declares its signatures.
There is no Python or CPU implementation behind these names: if the library is
missing, or no CUDA device is present when a handle is created, the call fails.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FMB_LIB_PATH") or os.path.join(_HERE, "libfmb.so")   # FMB_LIB_PATH: a tuning build, tools/ only

FMB_OK = 0
FMB_ERR_ARG, FMB_ERR_UNSUPPORTED, FMB_ERR_CUDA, FMB_ERR_NOMEM, FMB_ERR_STATE, FMB_ERR_IO = -1, -2, -3, -4, -5, -6
FMB_REF_BLOCK_BYTES = 262144
FMB_BLOCK_QUANTUM = 32768
FMB_PRECISION_EXACT, FMB_PRECISION_FMA = 0, 1
FMB_PIPE_DEPTH = 3
FMB_HIST = 128

class FmbConfig(C.Structure):
    """struct fmb_config (include/fmb.h) == the demod_state fields that fix numerics."""
    _fields_ = [
        ("rate_in", C.c_int), ("rate_out2", C.c_int), ("mode", C.c_int), ("size", C.c_int),
        ("offset_tuning", C.c_int), ("deemph", C.c_double), ("volume", C.c_float),
        ("n_streams", C.c_int), ("block_bytes", C.c_int), ("device", C.c_int),
        ("precision", C.c_int), ("segments", C.c_int), ("emulate_inplace_quirk", C.c_int),
        ("deemph_lambda", C.c_float), ("rate_out", C.c_int), ("max_blocks_per_call", C.c_int),
    ]


class FmbStreamState(C.Structure):
    """struct fmb_stream_state (include/fmb.h)."""
    _fields_ = [
        ("lowpass_tb", C.c_float * 48), ("pre_r", C.c_float), ("pre_j", C.c_float),
        ("br", C.c_float * FMB_HIST), ("bm", C.c_float * FMB_HIST), ("bs", C.c_float * FMB_HIST),
        ("pp", C.c_float), ("deemph_l", C.c_float), ("deemph_r", C.c_float), ("raw_valid", C.c_int),
        ("reserved", C.c_float * 2), ("raw_tail", C.c_ubyte * 64),
    ]


class FmbError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str):
        super().__init__(f"{where} failed with {code}: {detail}")
        self.code = code


_lib = None

# name -> (restype, argtypes); every symbol include/fmb.h declares
SIGNATURES = {
    "fmb_default_config": (C.c_int, [C.POINTER(FmbConfig)]),
    "fmb_preset_stereo_192k": (C.c_int, [C.POINTER(FmbConfig)]),
    "fmb_preset_mono_192k": (C.c_int, [C.POINTER(FmbConfig)]),
    "fmb_create": (C.c_int, [C.POINTER(FmbConfig), C.POINTER(C.c_void_p)]),
    "fmb_destroy": (C.c_int, [C.c_void_p]),
    "fmb_reset": (C.c_int, [C.c_void_p]),
    "fmb_set_volume": (C.c_int, [C.c_void_p, C.c_float]),
    "fmb_next_out_count": (C.c_int, [C.c_void_p]),
    "fmb_set_blocks_per_call": (C.c_int, [C.c_void_p, C.c_int]),
    "fmb_out_count_blocks": (C.c_int, [C.c_void_p, C.c_int]),
    "fmb_max_out_count": (C.c_int, [C.c_void_p]),
    "fmb_process": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "fmb_process_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "fmb_join": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fmb_input_ready": (C.c_int, [C.c_void_p]),
    "fmb_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "fmb_wait": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "fmb_bind_thread_to_device_node": (C.c_int, [C.c_int]),
    "fmb_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "fmb_host_alloc_wc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "fmb_host_free": (C.c_int, [C.c_void_p]),
    "fmb_get_state": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(FmbStreamState), C.POINTER(C.c_int),
                                C.POINTER(C.c_uint64)]),
    "fmb_set_state": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(FmbStreamState), C.c_int, C.c_uint64]),
    "fmb_get_tables": (C.c_int, [C.c_void_p] + [C.POINTER(C.c_float)] * 5),
    "fmb_debug_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "fmb_debug_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    "fmb_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "fmb_profile_reset": (C.c_int, [C.c_void_p]),
    "fmb_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "fmb_deemph_fallbacks": (C.c_int, [C.c_void_p, C.POINTER(C.c_ulonglong)]),
    "fmb_last_error": (C.c_char_p, []),
    "fmb_launch_count": (C.c_long, []),
    "fmb_version": (C.c_char_p, []),
    "fmb_internal_stream": (C.c_void_p, [C.c_void_p]),
    "fmb_sync": (C.c_int, [C.c_void_p]),
    "fmb_demod_kernel_name": (C.c_char_p, [C.c_void_p]),
    "fmb_deemph_kernel_name": (C.c_char_p, [C.c_void_p]),
    "fmb_set_stream_output": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_double),
                                        C.POINTER(C.c_float)]),
    "fmb_get_stream_output": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                        C.POINTER(C.c_int)]),
    # include/fmb_multi.h: the C multi-GPU host (one worker thread per device)
    "fmb_multi_create": (C.c_int, [C.POINTER(FmbConfig), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "fmb_multi_destroy": (C.c_int, [C.c_void_p]),
    "fmb_multi_shards": (C.c_int, [C.c_void_p]),
    "fmb_multi_shard_range": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "fmb_multi_handle": (C.c_void_p, [C.c_void_p, C.c_int]),
    "fmb_multi_next_out_count": (C.c_int, [C.c_void_p]),
    "fmb_multi_set_blocks_per_call": (C.c_int, [C.c_void_p, C.c_int]),
    "fmb_multi_out_count_blocks": (C.c_int, [C.c_void_p, C.c_int]),
    "fmb_multi_max_out_count": (C.c_int, [C.c_void_p]),
    "fmb_multi_reset": (C.c_int, [C.c_void_p]),
    "fmb_multi_set_stream_output": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float),
                                              C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "fmb_multi_get_stream_output": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float),
                                              C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "fmb_multi_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "fmb_multi_wait": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "fmb_multi_process": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "fmb_multi_process_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_size_t, C.POINTER(C.c_void_p), C.c_size_t]),
    "fmb_multi_sync": (C.c_int, [C.c_void_p]),
    "fmb_parse_device_list": (C.c_int, [C.c_char_p, C.POINTER(C.c_int), C.c_int]),
    "fmb_device_count": (C.c_int, []),
}


def build(verbose: bool = False) -> str:
    """Compile libfmb.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j4"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libfmb.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    if verbose:
        print(r.stdout[-2000:])
    return LIB_PATH


def lib() -> C.CDLL:
    """Load libfmb.so (once).  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C rtl_fm_player_b200/csrc`. There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def stream_output_args(n_streams: int, first: int, volume, deemph, deemph_lambda):
    """(count, volume, deemph, deemph_lambda) for fmb[_multi]_set_stream_output: each setting None (keep), a scalar
    broadcast over the range or an array of its length.  The range is [first, first + len) of the arrays given, or
    [first, n_streams) when every setting is a scalar."""
    import numpy as np
    given = [(v, t) for v, t in ((volume, np.float32), (deemph, np.float64), (deemph_lambda, np.float32))]
    lens = {np.size(v) for v, _ in given if v is not None and np.ndim(v) > 0}
    if len(lens) > 1:
        raise ValueError(f"per-stream settings of different lengths {sorted(lens)}")
    count = lens.pop() if lens else n_streams - first
    out = []
    for v, t in given:
        if v is None:
            out.append((None, None))
        else:
            a = np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=t), (count,)))
            ct = C.c_double if t is np.float64 else C.c_float
            out.append((a, a.ctypes.data_as(C.POINTER(ct))))
    # the arrays are returned with their pointers so that they outlive the call
    return count, out


def check(rc: int, where: str) -> int:
    if rc < 0:
        raise FmbError(rc, where, lib().fmb_last_error().decode(errors="replace"))
    return rc
