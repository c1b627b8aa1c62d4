"""ctypes access to the two CPU checkers.  TEST INFRASTRUCTURE ONLY.

  * `PortOracle`  -- oracle/libfm_oracle.so, our C restatement (oracle/fm_oracle.c); with fma=True
                     oracle/libfm_oracle_fma.so, the same built with FMO_FMA (FIR multiply-adds fused:
                     the definition of FMB_PRECISION_FMA)
  * `RefOracle`   -- oracle/_ref/libfmref.so, the reference's own rtl_fm_player.c compiled
                     unmodified (oracle/ref_harness.c); built only where /root/reference exists,
                     the prebuilt file travels to the GPU box.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  Nothing under rtl_fm_player_b200/ does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
PORT_PATH = os.path.join(_HERE, "libfm_oracle.so")
PORT_FMA_PATH = os.path.join(_HERE, "libfm_oracle_fma.so")
REF_PATH = os.path.join(_HERE, "_ref", "libfmref.so")
REF_CLI = os.path.join(_HERE, "_ref", "ref_offline")
REF_BLOCK = 262144


def build(which: str = "all") -> None:
    r = subprocess.run(["make", "-C", _HERE, which], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)


class _PortCfg(C.Structure):
    _fields_ = [("rate_in", C.c_int), ("rate_out2", C.c_int), ("mode", C.c_int), ("size", C.c_int),
                ("offset_tuning", C.c_int), ("deemph", C.c_double), ("volume", C.c_float), ("inplace_quirk", C.c_int),
                ("rate_out", C.c_int)]


class _RefCfg(C.Structure):
    _fields_ = [("rate_in", C.c_int), ("rate_out2", C.c_int), ("mode", C.c_int), ("size", C.c_int),
                ("offset_tuning", C.c_int), ("deemph", C.c_double), ("volume", C.c_float), ("rate_out", C.c_int)]


class PortState(C.Structure):
    _fields_ = [("tb", C.c_float * 48), ("pre_r", C.c_float), ("pre_j", C.c_float), ("br", C.c_float * 128),
                ("bm", C.c_float * 128), ("bs", C.c_float * 128), ("pp", C.c_float), ("deemph_l", C.c_float),
                ("deemph_r", C.c_float), ("reserved", C.c_float * 3)]


def _f32(n):
    return np.empty(max(n, 1), dtype=np.float32)


class PortOracle:
    """One channel of the C restatement; fma=True: its fused build, the model of FMB_PRECISION_FMA."""

    def __init__(self, rate_in=240000, rate_out2=48000, mode=2, size=90, offset_tuning=0, deemph=0.000050,
                 volume=0.4, inplace_quirk=1, rate_out=0, fma=False):
        path = PORT_FMA_PATH if fma else PORT_PATH
        if not os.path.exists(path):
            build("port")
        self.lib = C.CDLL(path)
        self.lib.fmo_create.restype = C.c_void_p
        self.lib.fmo_create.argtypes = [C.POINTER(_PortCfg)]
        self.lib.fmo_destroy.argtypes = [C.c_void_p]
        self.lib.fmo_block.restype = C.c_int
        self.lib.fmo_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 4
        self.lib.fmo_run.restype = C.c_long
        self.lib.fmo_run.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.c_size_t]
        self.lib.fmo_bench.restype = C.c_long
        self.lib.fmo_bench.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_int]
        self.lib.fmo_get_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        self.lib.fmo_get_state.argtypes = [C.c_void_p, C.POINTER(PortState), C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
        self.lib.fmo_set_state.argtypes = [C.c_void_p, C.POINTER(PortState), C.c_int, C.c_uint64]
        self.cfg = _PortCfg(rate_in, rate_out2, mode, size, offset_tuning, deemph, volume, inplace_quirk, rate_out)
        self.h = self.lib.fmo_create(C.byref(self.cfg))
        if not self.h:
            raise ValueError("fmo_create rejected the configuration")

    def __del__(self):
        try:
            if self.h:
                self.lib.fmo_destroy(self.h)
        except Exception:
            pass

    def block(self, iq: np.ndarray, stages: bool = False):
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        n_dem = iq.size // 16
        pcm = np.empty(max(n_dem, 1), dtype=np.int16)
        if stages:
            dem, lr, de = _f32(n_dem), _f32(n_dem), _f32(n_dem)
            n = self.lib.fmo_block(self.h, iq.ctypes.data, iq.size, pcm.ctypes.data, dem.ctypes.data, lr.ctypes.data,
                                   de.ctypes.data)
            return pcm[:n].copy(), {"dem": dem[:n_dem].copy(), "lr": lr[:n].copy(), "de": de[:n].copy()}
        n = self.lib.fmo_block(self.h, iq.ctypes.data, iq.size, pcm.ctypes.data, None, None, None)
        return pcm[:n].copy()

    def run(self, iq: np.ndarray, block_bytes: int = REF_BLOCK) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        cap = iq.size // 16 + 16
        pcm = np.empty(cap, dtype=np.int16)
        n = self.lib.fmo_run(self.h, iq.ctypes.data, iq.size, block_bytes, pcm.ctypes.data, cap)
        assert n >= 0
        return pcm[:n].copy()

    def bench(self, iq: np.ndarray, repeat: int, block_bytes: int = REF_BLOCK) -> int:
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        return int(self.lib.fmo_bench(self.h, iq.ctypes.data, iq.size, block_bytes, repeat))

    def tables(self):
        taps = self.cfg.size // 2
        fb, fm, fp, fs, misc = _f32(16), _f32(taps), _f32(taps), _f32(taps), _f32(4)
        self.lib.fmo_get_tables(self.h, *(a.ctypes.data for a in (fb, fm, fp, fs, misc)))
        return {"fb": fb, "fm": fm, "fp": fp, "fs": fs, "misc": misc}

    def state(self):
        st, ph, bl = PortState(), C.c_int(0), C.c_uint64(0)
        self.lib.fmo_get_state(self.h, C.byref(st), C.byref(ph), C.byref(bl))
        return st, ph.value, bl.value

    def set_state(self, st: PortState, phase: int, blocks: int) -> None:
        self.lib.fmo_set_state(self.h, C.byref(st), phase, blocks)


def ref_available() -> bool:
    return os.path.exists(REF_PATH)


class RefOracle:
    """One channel of the reference's own code (oracle/_ref/libfmref.so)."""

    def __init__(self, rate_in=240000, rate_out2=48000, mode=2, size=90, offset_tuning=0, deemph=0.000050, volume=0.4,
                 rate_out=0):
        if not ref_available():
            raise FileNotFoundError(REF_PATH)
        self.lib = C.CDLL(REF_PATH)
        self.lib.ref_create.restype = C.c_void_p
        self.lib.ref_create.argtypes = [C.POINTER(_RefCfg)]
        self.lib.ref_destroy.argtypes = [C.c_void_p]
        self.lib.ref_block.restype = C.c_int
        self.lib.ref_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        self.lib.ref_block_stages.restype = C.c_int
        self.lib.ref_block_stages.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 6
        self.lib.ref_run.restype = C.c_long
        self.lib.ref_run.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        self.lib.ref_get_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        self.lib.ref_layout.restype = C.c_long
        self.lib.ref_layout.argtypes = [C.c_int]
        self.cfg = _RefCfg(rate_in, rate_out2, mode, size, offset_tuning, deemph, volume, rate_out)
        self.h = self.lib.ref_create(C.byref(self.cfg))

    def __del__(self):
        try:
            if self.h:
                self.lib.ref_destroy(self.h)
        except Exception:
            pass

    def block(self, iq: np.ndarray, stages: bool = False):
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        assert iq.size <= REF_BLOCK
        pcm = np.empty(REF_BLOCK // 2, dtype=np.int16)
        if stages:
            z, dem, lr, de = _f32(iq.size // 8), _f32(iq.size // 16), _f32(iq.size // 16), _f32(iq.size // 16)
            ns = (C.c_int * 2)()
            n = self.lib.ref_block_stages(self.h, iq.ctypes.data, iq.size, z.ctypes.data, dem.ctypes.data,
                                          lr.ctypes.data, de.ctypes.data, pcm.ctypes.data, ns)
            return pcm[:n].copy(), {"z": z[:ns[0]].copy(), "dem": dem[:ns[1]].copy(), "lr": lr[:n].copy(),
                                    "de": de[:n].copy()}
        n = self.lib.ref_block(self.h, iq.ctypes.data, iq.size, pcm.ctypes.data)
        return pcm[:n].copy()

    def run(self, iq: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        cap = iq.size // 16 + 16
        pcm = np.empty(cap, dtype=np.int16)
        n = self.lib.ref_run(self.h, iq.ctypes.data, iq.size, pcm.ctypes.data, cap)
        assert n >= 0
        return pcm[:n].copy()

    def tables(self):
        taps = self.cfg.size // 2
        fb, fm, fp, fs, misc = _f32(16), _f32(taps), _f32(taps), _f32(taps), _f32(3)
        self.lib.ref_get_tables(self.h, *(a.ctypes.data for a in (fb, fm, fp, fs, misc)))
        return {"fb": fb, "fm": fm, "fp": fp, "fs": fs, "misc": misc}

    def layout(self, what: int) -> int:
        return int(self.lib.ref_layout(what))
