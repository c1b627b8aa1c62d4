"""Host-side mirror of the reference's demod interface for a BATCH of channels.

`FmBatch` plays the role of the reference's `struct demod_state` + `full_demod`
(src/rtl_fm_player.c:758-788, include/rtl_fm_player.h:127-175) for n_streams
independent FM channels: configure it with the same fields (`rate_in`,
`rate_out2`, `lpr.mode`, `lpr.size`, `offset_tuning`, `deemph`, `volume`), feed it
one uint8 IQ block per stream per call, get that block's int16 PCM per stream.
All work happens in libfmb.so's CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib as L


@dataclass
class DemodConfig:
    """The demod_state fields that fix numerics; defaults = demod_init (:1156-1195)."""
    rate_in: int = 240000
    rate_out2: int = 48000
    mode: int = 2
    size: int = 90
    offset_tuning: int = 0
    deemph: float = 0.000050
    volume: float = 0.4
    n_streams: int = 1
    block_bytes: int = L.FMB_REF_BLOCK_BYTES
    device: int = 0
    precision: int = L.FMB_PRECISION_EXACT
    segments: int = 0
    emulate_inplace_quirk: int = 1
    deemph_lambda: float = 0.0
    rate_out: int = 0          # demod.rate_out (the resampler's fast rate, :485); 0 = rate_in
    max_blocks_per_call: int = 0   # most consecutive blocks per stream one call may take; 0 = 1

    @classmethod
    def stereo_192k(cls, **kw) -> "DemodConfig":
        """The -X preset (:1464-1476)."""
        return cls(rate_in=192000, rate_out2=48000, mode=2, size=90, **kw)

    @classmethod
    def mono_192k(cls, **kw) -> "DemodConfig":
        """The -Y preset (:1477-1488)."""
        return cls(rate_in=192000, rate_out2=48000, mode=1, size=128, **kw)

    def to_c(self) -> L.FmbConfig:
        c = L.FmbConfig()
        for f, _ in L.FmbConfig._fields_:
            setattr(c, f, getattr(self, f))
        return c

    @property
    def channels(self) -> int:
        return 2 if self.mode == 2 else 1

    @property
    def iq_samples_per_block(self) -> int:
        return self.block_bytes // 2

    @property
    def max_blocks(self) -> int:
        return max(1, self.max_blocks_per_call)


class FmBatch:
    """n_streams demodulators behind one handle (fmb_create / fmb_process / fmb_destroy)."""

    def __init__(self, cfg: DemodConfig):
        self.cfg = cfg
        self._lib = L.lib()
        self._h = C.c_void_p()
        cc = cfg.to_c()
        L.check(self._lib.fmb_create(C.byref(cc), C.byref(self._h)), "fmb_create")
        self.max_out = self._lib.fmb_max_out_count(self._h)
        self._blocks = cfg.max_blocks          # blocks per call, as fmb_create leaves it
        self._last_blocks = 1

    # -- lifetime ---------------------------------------------------------------------------
    def close(self) -> None:
        if self._h:
            self._lib.fmb_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- queries ----------------------------------------------------------------------------
    def next_out_count(self) -> int:
        return L.check(self._lib.fmb_next_out_count(self._h), "fmb_next_out_count")

    def set_blocks_per_call(self, n: int) -> None:
        """Blocks per stream the following calls consume (1 .. max_blocks_per_call; default the maximum)."""
        L.check(self._lib.fmb_set_blocks_per_call(self._h, n), "fmb_set_blocks_per_call")
        self._blocks = n

    def out_count_blocks(self, n_blocks: int) -> int:
        """int16 values per stream the first n_blocks blocks of the next call produce."""
        return L.check(self._lib.fmb_out_count_blocks(self._h, n_blocks), "fmb_out_count_blocks")

    def kernel_name(self) -> str:
        return self._lib.fmb_demod_kernel_name(self._h).decode()

    def deemph_kernel_name(self) -> str:
        """The de-emphasis kernel the next call launches (fmb_deemph_kernel_name)."""
        return self._lib.fmb_deemph_kernel_name(self._h).decode()

    def set_volume(self, volume: float) -> None:
        """Volume of every stream (fmb_set_volume)."""
        L.check(self._lib.fmb_set_volume(self._h, volume), "fmb_set_volume")

    def set_stream_output(self, volume=None, deemph=None, deemph_lambda=None, first: int = 0) -> None:
        """Output settings of streams [first, first + n) from the next call on (fmb_set_stream_output): volume,
        de-emphasis time constant in seconds (0 = off) and pole override (> 0).  None keeps a setting; a scalar is
        broadcast over the range, an array gives one value per stream and n is its length (with scalars only, the
        range runs to the last stream)."""
        count, args = L.stream_output_args(self.cfg.n_streams, first, volume, deemph, deemph_lambda)
        L.check(self._lib.fmb_set_stream_output(self._h, first, count, *(p for _, p in args)), "fmb_set_stream_output")

    def stream_output(self, first: int = 0, count: int | None = None) -> dict:
        """{"volume", "lambda", "deemph_on"} of streams [first, first + count) (fmb_get_stream_output)."""
        count = self.cfg.n_streams - first if count is None else count
        vol, lam, on = (np.empty(count, np.float32), np.empty(count, np.float32), np.empty(count, np.int32))
        L.check(self._lib.fmb_get_stream_output(self._h, first, count, vol.ctypes.data_as(C.POINTER(C.c_float)),
                                                lam.ctypes.data_as(C.POINTER(C.c_float)),
                                                on.ctypes.data_as(C.POINTER(C.c_int))), "fmb_get_stream_output")
        return {"volume": vol, "lambda": lam, "deemph_on": on.astype(bool)}

    def reset(self) -> None:
        L.check(self._lib.fmb_reset(self._h), "fmb_reset")

    def tables(self):
        taps = self.cfg.size // 2
        fb = (C.c_float * 16)()
        fm, fp, fs = ((C.c_float * taps)() for _ in range(3))
        misc = (C.c_float * 4)()
        L.check(self._lib.fmb_get_tables(self._h, fb, fm, fp, fs, misc), "fmb_get_tables")
        f = lambda a: np.frombuffer(a, dtype=np.float32).copy()
        return {"fb": f(fb), "fm": f(fm), "fp": f(fp), "fs": f(fs), "misc": f(misc)}

    # -- host path (the drop-in granularity: one block per stream in, PCM out) --------------
    def process(self, iq: np.ndarray) -> np.ndarray:
        """iq: uint8 [n_streams, m * block_bytes], 1 <= m <= max_blocks_per_call, m consecutive blocks of each
        stream -> int16 [n_streams, n_out] (fmb_process), the concatenation of the m blocks' PCM."""
        m = iq.shape[1] // self.cfg.block_bytes if iq.ndim == 2 else 0
        if m != self._blocks and 1 <= m <= self.cfg.max_blocks:
            self.set_blocks_per_call(m)
        iq = self._check_iq(iq)
        n = self.next_out_count()
        pitch = max(8, (n + 7) & ~7)
        pcm = np.empty((self.cfg.n_streams, pitch), dtype=np.int16)
        row = m * self.cfg.block_bytes
        iq_pitch = iq.strides[0] if iq.shape[0] > 1 else row   # a 1-row view may carry stride 0
        L.check(self._lib.fmb_process(self._h, iq.ctypes.data, iq_pitch, pcm.ctypes.data, pitch, None),
                "fmb_process")
        self._last_blocks = m
        return pcm[:, :n]

    def run(self, iq: np.ndarray) -> np.ndarray:
        """Whole captures: uint8 [n_streams, n_bytes]; full blocks only, the short tail is
        dropped as demod_thread_fn does (:863-868).  Calls of max_blocks_per_call blocks, and a shorter
        last one.  Returns int16 [n_streams, total]."""
        assert iq.ndim == 2 and iq.shape[0] == self.cfg.n_streams
        bb, k = self.cfg.block_bytes, self.cfg.max_blocks
        n_blocks = iq.shape[1] // bb
        outs = [self.process(iq[:, b * bb:min(b + k, n_blocks) * bb]) for b in range(0, n_blocks, k)]
        if not outs:
            return np.empty((self.cfg.n_streams, 0), dtype=np.int16)
        return np.concatenate(outs, axis=1)

    def submit(self, iq_ptr: int, iq_pitch: int, pcm_ptr: int, pcm_pitch: int) -> int:
        t = C.c_int(-1)
        L.check(self._lib.fmb_submit(self._h, iq_ptr, iq_pitch, pcm_ptr, pcm_pitch, C.byref(t)), "fmb_submit")
        return t.value

    def wait(self, ticket: int) -> None:
        L.check(self._lib.fmb_wait(self._h, ticket, None), "fmb_wait")

    # -- device-resident path -----------------------------------------------------------------
    def process_device(self, iq_ptr: int, iq_pitch: int, pcm_ptr: int, pcm_pitch: int, stream: int = 0) -> None:
        L.check(self._lib.fmb_process_device(self._h, iq_ptr, iq_pitch, pcm_ptr, pcm_pitch, stream),
                "fmb_process_device")

    def input_ready(self) -> None:
        """The next process_device() step waits for everything enqueued on its stream, kernels included."""
        L.check(self._lib.fmb_input_ready(self._h), "fmb_input_ready")

    def join(self, stream: int = 0) -> None:
        L.check(self._lib.fmb_join(self._h, stream), "fmb_join")

    # -- state / debug / profile ------------------------------------------------------------------
    def get_state(self, first: int = 0, count: int | None = None):
        count = self.cfg.n_streams - first if count is None else count
        arr = (L.FmbStreamState * count)()
        phase, blocks = C.c_int(0), C.c_uint64(0)
        L.check(self._lib.fmb_get_state(self._h, first, count, arr, C.byref(phase), C.byref(blocks)), "fmb_get_state")
        return arr, phase.value, blocks.value

    def set_state(self, arr, phase: int, blocks: int, first: int = 0) -> None:
        L.check(self._lib.fmb_set_state(self._h, first, len(arr), arr, phase, blocks), "fmb_set_state")

    def debug_enable(self, on: bool = True) -> None:
        L.check(self._lib.fmb_debug_enable(self._h, int(on)), "fmb_debug_enable")

    def debug_read(self):
        """Discriminator and decoder outputs of the last call (its whole rows)."""
        n_dem = self._last_blocks * self.cfg.block_bytes // 16
        dem = np.empty((self.cfg.n_streams, n_dem), dtype=np.float32)
        lr = np.empty((self.cfg.n_streams, max(self.max_out, 1)), dtype=np.float32)
        L.check(self._lib.fmb_debug_read(self._h, dem.ctypes.data, n_dem, lr.ctypes.data, lr.shape[1]), "fmb_debug_read")
        return dem, lr

    def deemph_fallbacks(self) -> int:
        """De-emphasis chunks whose time-speculation failed verification and were redone in order."""
        n = C.c_ulonglong(0)
        L.check(self._lib.fmb_deemph_fallbacks(self._h, C.byref(n)), "fmb_deemph_fallbacks")
        return int(n.value)

    def profile_enable(self, on: bool = True) -> None:
        L.check(self._lib.fmb_profile_enable(self._h, int(on)), "fmb_profile_enable")

    def profile_reset(self) -> None:
        L.check(self._lib.fmb_profile_reset(self._h), "fmb_profile_reset")

    def profile_read(self):
        ms = (C.c_double * 2)()
        n = (C.c_int * 2)()
        L.check(self._lib.fmb_profile_read(self._h, ms, n), "fmb_profile_read")
        return {"demod_ms": ms[0], "deemph_ms": ms[1], "demod_launches": n[0], "deemph_launches": n[1]}

    # -- helpers --------------------------------------------------------------------------------
    def _check_iq(self, iq: np.ndarray) -> np.ndarray:
        row = self._blocks * self.cfg.block_bytes
        if iq.dtype != np.uint8 or iq.ndim != 2 or iq.shape != (self.cfg.n_streams, row):
            raise ValueError(f"iq must be uint8 [{self.cfg.n_streams}, m * {self.cfg.block_bytes}] with "
                             f"1 <= m <= {self.cfg.max_blocks}, got {iq.dtype} {iq.shape}")
        if iq.strides[1] != 1 or (iq.shape[0] > 1 and (iq.strides[0] < row or iq.strides[0] % 16)) or iq.ctypes.data % 16:
            iq = np.ascontiguousarray(iq)       # (also a 1-stream view made with iq[None, ...] has stride 0)
            if iq.ctypes.data % 16:
                buf = np.empty(iq.size + 16, dtype=np.uint8)
                off = (-buf.ctypes.data) % 16
                aligned = buf[off:off + iq.size].reshape(iq.shape)
                aligned[...] = iq
                iq = aligned
        return iq


def launch_count() -> int:
    """CUDA kernels launched by libfmb.so in this process (fmb_launch_count)."""
    return int(L.lib().fmb_launch_count())
