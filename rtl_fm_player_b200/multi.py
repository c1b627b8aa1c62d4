"""ctypes mirror of include/fmb_multi.h: one batch of channels sharded over several GPUs by the C host
(one worker thread per device, csrc/fmb_multi.c).  The counterpart, per device, of the reference's demod
thread (src/rtl_fm_player.c:855-933).  All work happens in libfmb.so."""
from __future__ import annotations

import ctypes as C
from typing import List, Sequence, Tuple

import numpy as np

from . import _lib as L
from .batch import DemodConfig


def parse_device_list(text: str) -> List[int]:
    """"0-3,6" -> [0, 1, 2, 3, 6] (fmb_parse_device_list)."""
    out = (C.c_int * 64)()
    n = L.check(L.lib().fmb_parse_device_list(text.encode(), out, 64), "fmb_parse_device_list")
    return list(out[:n])


def device_count() -> int:
    return int(L.lib().fmb_device_count())


def pinned_array(shape: Tuple[int, ...], dtype, write_combined: bool = False) -> np.ndarray:
    """A numpy view of portable pinned host memory (fmb_host_alloc[_wc]); every device can DMA to/from it.
    The memory is freed when the returned array (the owner of the view chain) is garbage collected."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = C.c_void_p()
    fn = L.lib().fmb_host_alloc_wc if write_combined else L.lib().fmb_host_alloc
    L.check(fn(C.byref(ptr), max(nbytes, 16)), "fmb_host_alloc")
    raw = (C.c_uint8 * max(nbytes, 16)).from_address(ptr.value)
    arr = np.frombuffer(raw, dtype=np.uint8, count=nbytes).view(dtype).reshape(shape)

    class _Owner:
        def __init__(self, p): self.p = p
        def __del__(self):
            try:
                L.lib().fmb_host_free(self.p)
            except Exception:
                pass
    _KEEP[arr.ctypes.data] = _Owner(ptr)
    return arr


_KEEP: dict = {}


def free_pinned(arr: np.ndarray) -> None:
    _KEEP.pop(arr.ctypes.data, None)


class FmMulti:
    """cfg.n_streams channels over `devices` (fmb_multi_create / submit / wait / destroy)."""

    def __init__(self, cfg: DemodConfig, devices: Sequence[int]):
        self.cfg = cfg
        self._lib = L.lib()
        self._m = C.c_void_p()
        cc = cfg.to_c()
        dv = (C.c_int * len(devices))(*devices)
        L.check(self._lib.fmb_multi_create(C.byref(cc), dv, len(devices), C.byref(self._m)), "fmb_multi_create")
        self.max_out = self._lib.fmb_multi_max_out_count(self._m)
        self._blocks = cfg.max_blocks
        self.shards = []
        for g in range(self._lib.fmb_multi_shards(self._m)):
            first, count, dev = C.c_int(), C.c_int(), C.c_int()
            L.check(self._lib.fmb_multi_shard_range(self._m, g, C.byref(first), C.byref(count), C.byref(dev)),
                    "fmb_multi_shard_range")
            self.shards.append((first.value, count.value, dev.value))

    def close(self) -> None:
        if self._m:
            self._lib.fmb_multi_destroy(self._m)
            self._m = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def next_out_count(self) -> int:
        return L.check(self._lib.fmb_multi_next_out_count(self._m), "fmb_multi_next_out_count")

    def set_blocks_per_call(self, n: int) -> None:
        L.check(self._lib.fmb_multi_set_blocks_per_call(self._m, n), "fmb_multi_set_blocks_per_call")
        self._blocks = n

    def out_count_blocks(self, n_blocks: int) -> int:
        return L.check(self._lib.fmb_multi_out_count_blocks(self._m, n_blocks), "fmb_multi_out_count_blocks")

    def reset(self) -> None:
        L.check(self._lib.fmb_multi_reset(self._m), "fmb_multi_reset")

    def set_stream_output(self, volume=None, deemph=None, deemph_lambda=None, first: int = 0) -> None:
        """FmBatch.set_stream_output over global stream indices (fmb_multi_set_stream_output)."""
        count, args = L.stream_output_args(self.cfg.n_streams, first, volume, deemph, deemph_lambda)
        L.check(self._lib.fmb_multi_set_stream_output(self._m, first, count, *(p for _, p in args)),
                "fmb_multi_set_stream_output")

    def stream_output(self, first: int = 0, count: int | None = None) -> dict:
        """FmBatch.stream_output over global stream indices (fmb_multi_get_stream_output)."""
        count = self.cfg.n_streams - first if count is None else count
        vol, lam, on = (np.empty(count, np.float32), np.empty(count, np.float32), np.empty(count, np.int32))
        L.check(self._lib.fmb_multi_get_stream_output(self._m, first, count, vol.ctypes.data_as(C.POINTER(C.c_float)),
                                                      lam.ctypes.data_as(C.POINTER(C.c_float)),
                                                      on.ctypes.data_as(C.POINTER(C.c_int))), "fmb_multi_get_stream_output")
        return {"volume": vol, "lambda": lam, "deemph_on": on.astype(bool)}

    def deemph_kernel_name(self, shard: int = 0) -> str:
        """The de-emphasis kernel shard `shard`'s next call launches (fmb_deemph_kernel_name)."""
        return self._lib.fmb_deemph_kernel_name(self.shard_handle(shard)).decode()

    def shard_handle(self, g: int) -> int:
        return self._lib.fmb_multi_handle(self._m, g)

    def submit(self, iq_ptr: int, iq_pitch: int, pcm_ptr: int, pcm_pitch: int) -> int:
        t = C.c_int(-1)
        L.check(self._lib.fmb_multi_submit(self._m, iq_ptr, iq_pitch, pcm_ptr, pcm_pitch, C.byref(t)), "fmb_multi_submit")
        return t.value

    def wait(self, ticket: int) -> None:
        L.check(self._lib.fmb_multi_wait(self._m, ticket, None), "fmb_multi_wait")

    def process(self, iq: np.ndarray, pcm: np.ndarray | None = None) -> np.ndarray:
        """iq: uint8 [n_streams, m * block_bytes], 1 <= m <= max_blocks_per_call (ideally pinned_array)
        -> int16 [n_streams, n_out]."""
        S = self.cfg.n_streams
        m = iq.shape[1] // self.cfg.block_bytes
        if m != self._blocks:
            self.set_blocks_per_call(m)
        B = m * self.cfg.block_bytes
        assert iq.dtype == np.uint8 and iq.shape == (S, B) and iq.flags.c_contiguous and iq.ctypes.data % 16 == 0
        n = self.next_out_count()
        pitch = max(8, (n + 7) & ~7)
        if pcm is None:
            pcm = np.empty((S, pitch), dtype=np.int16)
        assert pcm.dtype == np.int16 and pcm.shape[0] == S and pcm.shape[1] >= n and pcm.flags.c_contiguous
        n_out = (C.c_int * S)()
        L.check(self._lib.fmb_multi_process(self._m, iq.ctypes.data, B, pcm.ctypes.data, pcm.shape[1], n_out),
                "fmb_multi_process")
        assert all(v == n for v in n_out)
        return pcm[:, :n]

    def run(self, iq: np.ndarray) -> np.ndarray:
        """Whole captures uint8 [n_streams, n_bytes]; full blocks only (demod_thread_fn :863-868)."""
        S, B, k = self.cfg.n_streams, self.cfg.block_bytes, self.cfg.max_blocks
        n_blocks = iq.shape[1] // B
        stage = pinned_array((S, k * B), np.uint8)
        outs = []
        try:
            for b in range(0, n_blocks, k):
                m = min(k, n_blocks - b)
                st = stage[:, :m * B] if m == k else np.ascontiguousarray(stage[:, :m * B])
                st[...] = iq[:, b * B:(b + m) * B]
                outs.append(self.process(st).copy())
        finally:
            free_pinned(stage)
        return np.concatenate(outs, axis=1) if outs else np.empty((S, 0), dtype=np.int16)

    def process_device(self, iq_ptrs: Sequence[int], iq_pitch: int, pcm_ptrs: Sequence[int], pcm_pitch: int) -> None:
        a = (C.c_void_p * len(iq_ptrs))(*iq_ptrs)
        b = (C.c_void_p * len(pcm_ptrs))(*pcm_ptrs)
        L.check(self._lib.fmb_multi_process_device(self._m, a, iq_pitch, b, pcm_pitch), "fmb_multi_process_device")

    def sync(self) -> None:
        L.check(self._lib.fmb_multi_sync(self._m), "fmb_multi_sync")
