"""CPU tests of the host-side C pieces that replace the reference's I/O plumbing:
the file source with the rtlsdr_read_async contract (include/fm_filesrc.h), the WAV writer
(include/fm_wav.h) and the struct-offset header of the drop-in shim (csrc/ref_layout.h)."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import threading
import time

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from vectors import CONFIGS, make_input

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libfmref.so")
REF_SRC = "/root/reference/src/rtl_fm_player.c"
CB = C.CFUNCTYPE(None, C.POINTER(C.c_ubyte), C.c_uint32, C.c_void_p)



def lib():
    L = C.CDLL(R.LIB_PATH)
    L.filesrc_open.argtypes = [C.POINTER(C.c_void_p), C.c_char_p]
    L.filesrc_close.argtypes = [C.c_void_p]
    L.filesrc_read_async.argtypes = [C.c_void_p, CB, C.c_void_p, C.c_uint32, C.c_uint32]
    L.filesrc_cancel_async.argtypes = [C.c_void_p]
    L.filesrc_set_backpressure.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.c_uint32]
    L.filesrc_set_realtime.argtypes = [C.c_void_p, C.c_double]
    L.filesrc_set_sample_rate.argtypes = [C.c_void_p, C.c_uint32]
    L.filesrc_set_loop.argtypes = [C.c_void_p, C.c_uint32]
    L.filesrc_read_sync.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    L.filesrc_bytes_delivered.restype = C.c_uint64
    L.filesrc_bytes_delivered.argtypes = [C.c_void_p]
    L.filesrc_chunks_delivered.restype = C.c_uint64
    L.filesrc_chunks_delivered.argtypes = [C.c_void_p]
    L.fm_wav_open.argtypes = [C.POINTER(C.c_void_p), C.c_char_p, C.c_int]
    L.fm_wav_write.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.fm_wav_keep_tail.argtypes = [C.c_void_p, C.c_int]
    L.fm_wav_close.argtypes = [C.c_void_p]
    L.fm_wav_header.argtypes = [C.c_int, C.c_void_p]
    return L


def open_src(L, path):
    d = C.c_void_p()
    assert L.filesrc_open(C.byref(d), str(path).encode()) == 0
    return d


def test_filesrc_delivers_whole_chunks_in_order_and_drops_the_tail(tmp_path):
    L = lib()
    data = np.random.default_rng(1).integers(0, 256, 3 * 262144 + 49152, dtype=np.uint8)
    p = tmp_path / "cap.u8"
    data.tofile(p)
    got = []
    cb = CB(lambda buf, n, ctx: got.append(bytes(C.cast(buf, C.POINTER(C.c_ubyte * n)).contents)))
    d = open_src(L, p)
    assert L.filesrc_read_async(d, cb, None, 0, 0) == 0          # buf_len 0 -> 262144 (librtlsdr.c:354-355)
    assert [len(g) for g in got] == [262144] * 3                   # 49152-byte tail never delivered (:863-868)
    assert b"".join(got) == data[:3 * 262144].tobytes()
    assert L.filesrc_bytes_delivered(d) == 3 * 262144 and L.filesrc_chunks_delivered(d) == 3
    L.filesrc_close(d)
    d = open_src(L, p)
    assert L.filesrc_read_async(d, cb, None, 15, 1000) == -1     # not a multiple of 512 (rtl-sdr.h:366)
    L.filesrc_close(d)
    d = C.c_void_p()
    assert L.filesrc_open(C.byref(d), str(tmp_path / "missing").encode()) == -1


def test_filesrc_cancel_loop_and_sync_read(tmp_path):
    L = lib()
    data = np.arange(8 * 16384, dtype=np.uint32).view(np.uint8)     # 8 chunks of 65536
    p = tmp_path / "cap.u8"
    data.tofile(p)
    d = open_src(L, p)
    n = [0]

    def on_chunk(buf, ln, ctx):
        n[0] += 1
        if n[0] == 3:
            L.filesrc_cancel_async(d)                               # like rtlsdr_cancel_async from the callback (:795)
    cb = CB(on_chunk)
    assert L.filesrc_read_async(d, cb, None, 0, 65536) == 0
    assert n[0] == 3
    L.filesrc_close(d)
    d = open_src(L, p)
    L.filesrc_set_loop(d, 2)
    n[0] = -10 ** 9
    cnt = [0]
    cb2 = CB(lambda b, ln, c: cnt.__setitem__(0, cnt[0] + 1))
    assert L.filesrc_read_async(d, cb2, None, 0, 65536) == 0
    assert cnt[0] == 24
    L.filesrc_close(d)
    d = open_src(L, p)
    buf = np.zeros(100000, np.uint8)
    k = C.c_int(0)
    assert L.filesrc_read_sync(d, buf.ctypes.data, 100000, C.byref(k)) == 0 and k.value == 100000
    assert np.array_equal(buf, data[:100000])
    L.filesrc_close(d)


def test_filesrc_backpressure_never_overruns_the_consumers_ring(tmp_path):
    """The reference ring overwrites on overrun (rtl_fm_player.c:821-834); the file source waits."""
    L = lib()
    chunk, nchunks, ring_max = 16384, 40, 4 * 16384
    p = tmp_path / "cap.u8"
    np.zeros(chunk * nchunks, np.uint8).tofile(p)
    fill = C.c_uint32(0)
    lock = threading.Lock()
    peak = [0]

    def on_chunk(buf, ln, ctx):
        with lock:
            fill.value += ln
            peak[0] = max(peak[0], fill.value)
    cb = CB(on_chunk)
    d = open_src(L, p)
    L.filesrc_set_backpressure(d, C.byref(fill), ring_max)
    done = []
    t = threading.Thread(target=lambda: done.append(L.filesrc_read_async(d, cb, None, 0, chunk)))
    t.start()
    consumed = 0
    while consumed < nchunks:                                          # a slow consumer
        time.sleep(0.002)
        with lock:
            if fill.value >= chunk:
                fill.value -= chunk
                consumed += 1
    t.join(timeout=10)
    assert done == [0] and peak[0] <= ring_max and L.filesrc_chunks_delivered(d) == nchunks
    L.filesrc_close(d)


def test_filesrc_realtime_pacing(tmp_path):
    L = lib()
    p = tmp_path / "cap.u8"
    np.zeros(8 * 16384, np.uint8).tofile(p)                           # 65536 IQ samples
    d = open_src(L, p)
    L.filesrc_set_sample_rate(d, 1536000)
    L.filesrc_set_realtime(d, 0.25)                                  # 65536 / (1.536e6 * 0.25) = 0.17 s
    cb = CB(lambda b, n, c: None)
    t0 = time.perf_counter()
    assert L.filesrc_read_async(d, cb, None, 0, 16384) == 0
    dt = time.perf_counter() - t0
    assert 0.15 < dt < 1.0
    L.filesrc_close(d)


def _ref():
    if not os.path.exists(REF_SO):
        pytest.skip("oracle/_ref/libfmref.so not built (needs /root/reference)")
    Rf = C.CDLL(REF_SO)
    Rf.ref_wav_write.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_size_t]
    Rf.ref_wav_header.argtypes = [C.c_int, C.c_void_p]
    Rf.ref_layout.restype = C.c_long
    return Rf


@pytest.mark.parametrize("mode", [2, 1])
def test_wav_header_is_the_references(mode):
    L = lib()
    ours = (C.c_ubyte * 260)()
    assert L.fm_wav_header(mode, ours) == 0
    b = bytes(ours)
    # structural facts from include/rtl_fm_player.h:216-253
    assert b[:4] == b"RIFF" and b[8:16] == b"WAVEfmt " and b[36:40] == b"data" and b[44:] == bytes(216)
    assert int.from_bytes(b[22:24], "little") == (2 if mode == 2 else 1) and int.from_bytes(b[24:28], "little") == 48000
    golden = GOLDEN_WAV[f"header_{mode}"]
    assert hashlib.sha256(b).hexdigest() == golden
    if os.path.exists(REF_SO):                                        # and the live reference, where it is built
        theirs = (C.c_ubyte * 260)()
        assert _ref().ref_wav_header(mode, theirs) == 260
        assert bytes(theirs) == b


@pytest.mark.parametrize("mode,n_bytes", [(2, 1916928), (1, 958464), (2, 32768 * 3), (2, 1000), (1, 0)])
def test_wav_file_equals_the_references_byte_for_byte(tmp_path, mode, n_bytes):
    """config 2's shape: 117 blocks x 4096 frames x 4 B = 1916928 B of PCM -> 58 whole clusters in the file."""
    L = lib()
    pcm = np.random.default_rng(n_bytes + mode).integers(0, 256, n_bytes, dtype=np.uint8)
    ours = tmp_path / "ours.wav"
    w = C.c_void_p()
    assert L.fm_wav_open(C.byref(w), str(ours).encode(), mode) == 0
    for off in range(0, n_bytes, 16384 if mode == 2 else 8192):            # block-sized writes, like the demod thread
        part = pcm[off:off + (16384 if mode == 2 else 8192)]
        assert L.fm_wav_write(w, part.ctypes.data, part.size) == 0
    assert L.fm_wav_close(w) == 0
    data = ours.read_bytes()
    assert len(data) == 260 + (n_bytes // 32768) * 32768
    assert int.from_bytes(data[4:8], "little") == len(data) - 8 and int.from_bytes(data[40:44], "little") == len(data) - 44
    assert data[260:] == pcm[:(n_bytes // 32768) * 32768].tobytes()
    Rf = _ref()
    theirs = tmp_path / "theirs.wav"
    assert Rf.ref_wav_write(str(theirs).encode(), mode, pcm.ctypes.data, n_bytes) == 0
    assert theirs.read_bytes() == data


def test_wav_keep_tail_option(tmp_path):
    L = lib()
    pcm = np.arange(50000, dtype=np.uint8)
    p = tmp_path / "t.wav"
    w = C.c_void_p()
    assert L.fm_wav_open(C.byref(w), str(p).encode(), 2) == 0
    L.fm_wav_keep_tail(w, 1)
    L.fm_wav_write(w, pcm.ctypes.data, pcm.size)
    assert L.fm_wav_close(w) == 0
    assert p.read_bytes()[260:] == pcm.tobytes()


def _committed_layout():
    out = {}
    for line in open(os.path.join(ROOT, "rtl_fm_player_b200", "csrc", "ref_layout.h")):
        f = line.split()
        if len(f) == 3 and f[0] == "#define" and f[2].isdigit():
            out[f[1]] = int(f[2])
    return out


def test_dropin_layout_header_matches_the_reference_struct():
    lay = _committed_layout()
    assert lay["FMD_MAXIMUM_BUF_LENGTH"] == 262144
    L = lib()
    L.fm_dropin_sizeof_demod_state.restype = C.c_ulong
    assert L.fm_dropin_sizeof_demod_state() == lay["FMD_SIZEOF_DEMOD_STATE"]
    with open(os.path.join(HERE, "golden", "golden_meta.json")) as f:   # the reference's ref_layout(), recorded by
        ref = {int(k): v for k, v in json.load(f)["layout"].items()}  # tests/golden/make_golden.py
    for what, name in [(0, "FMD_SIZEOF_DEMOD_STATE"), (1, "FMD_OFF_buf"), (2, "FMD_OFF_buf_len"), (3, "FMD_OFF_lowpassed"),
                       (4, "FMD_OFF_lp_len"), (5, "FMD_OFF_lowpass_tb"), (6, "FMD_OFF_result"), (7, "FMD_OFF_result_len"),
                       (8, "FMD_OFF_offset_tuning"), (9, "FMD_OFF_rate_in"), (10, "FMD_OFF_rate_out"),
                       (11, "FMD_OFF_rate_out2"), (12, "FMD_OFF_pre_r_f32"), (13, "FMD_OFF_deemph"),
                       (14, "FMD_OFF_deemph_l_f32"), (15, "FMD_OFF_deemph_lambda"), (16, "FMD_OFF_volume"),
                       (17, "FMD_OFF_prev_lpr_index"), (18, "FMD_OFF_lpr"), (19, "FMD_OFF_rw"),
                       (20, "FMD_OFF_output_target"), (21, "FMD_SIZEOF_LP_REAL"), (25, "FMD_OFF_post_downsample")]:
        assert ref[what] == lay[name], name
    assert ref[22] == lay["FMD_LPR_OFF_swf"] and ref[23] == lay["FMD_LPR_OFF_pos"]
    assert ref[24] == lay["FMD_LPR_OFF_mode"]


@pytest.mark.skipif(not os.path.exists(REF_SRC), reason="the reference tree is only present in the authoring container")
def test_dropin_layout_header_is_fresh():
    gen = os.path.join(ROOT, "oracle", "_ref", "gen_layout")
    if not os.path.exists(gen):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], check=True, capture_output=True)
    out = subprocess.run([gen], capture_output=True, text=True, check=True).stdout
    assert out == open(os.path.join(ROOT, "rtl_fm_player_b200", "csrc", "ref_layout.h")).read()


# sha256 of the reference's 260-byte headers, from oracle/_ref/libfmref.so:ref_wav_header in the authoring container
GOLDEN_WAV = {'header_2': '37c5c07cffccd6f94a63c0cc58d6ce6e98f085193e2fbdf3a7b5ba2dba5ea48c', 'header_1': '7f3cfa10a8d1dff5fc794db3df826e2f92086088e2bd7df21d592acc46f87773'}


# ------------------------------------------------------------------------------------------
# timeshift ring (include/fm_timeshift.h) against a restatement of output_thread_fn's slot
# arithmetic, reference src/rtl_fm_player.c:962-1010
# ------------------------------------------------------------------------------------------
class RefTimeshift:
    """circbufferbotton / circbufferfull / circbufferout exactly as :945-1010 keeps them (one channel)."""

    def __init__(self, slots):
        self.slots, self.bottom, self.full, self.ring = slots, 0, 0, {}

    def push(self, cluster, shift):
        self.ring[self.bottom] = cluster                      # :964
        if shift < 0:                                         # :982
            shift = 0
        if self.full == 0:                                    # :985-987
            if shift > self.bottom:
                shift = self.bottom
        elif shift > self.slots - 2:                          # :988-991
            shift = self.slots - 2
        out = self.bottom - shift                             # :994
        if out < 0:                                           # :995-997
            out = self.slots - (shift - self.bottom)
        played = self.ring[out]                               # :1000 / :1004
        self.bottom += 1                                      # :1007-1010
        if self.bottom >= self.slots:
            self.full, self.bottom = 1, 0
        return out, shift, played


def _ts_lib():
    L = C.CDLL(R.LIB_PATH)
    L.fm_timeshift_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int]
    L.fm_timeshift_destroy.argtypes = [C.c_void_p]
    L.fm_timeshift_push.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.c_void_p]
    L.fm_timeshift_playback.argtypes = [C.c_void_p, C.c_int]
    L.fm_timeshift_playback.restype = C.c_void_p
    L.fm_timeshift_state.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.fm_timeshift_slots_for_kbytes.argtypes = [C.c_long]
    return L


def test_timeshift_slot_count_is_the_players():
    L = _ts_lib()
    assert L.fm_timeshift_slots_for_kbytes(180 * 1024) == 5760     # 180 MiB default, :1363-1364
    assert L.fm_timeshift_slots_for_kbytes(100) == 3
    ts = C.c_void_p()
    assert L.fm_timeshift_create(C.byref(ts), 1, 1) == -1 and L.fm_timeshift_create(C.byref(ts), 4, 0) == -1


@pytest.mark.parametrize("slots,n_streams", [(5, 1), (7, 3)])
def test_timeshift_ring_plays_what_the_reference_would(slots, n_streams):
    L = _ts_lib()
    CL = 32768
    rng = np.random.default_rng(slots)
    ts = C.c_void_p()
    assert L.fm_timeshift_create(C.byref(ts), slots, n_streams) == 0
    refs = [RefTimeshift(slots) for _ in range(n_streams)]
    shifts = [0, 0, 1, 3, 9, -2, 2, 2, 2, 100, 100, 0, 1, 4, 6, 5, 0, 3, 3, 3, 3, 3, 1]   # keyboard A/D/L walks
    out = np.empty((n_streams, CL), dtype=np.uint8)
    pitch = CL + 64                                                                       # padded producer rows
    for step, want_shift in enumerate(shifts):
        batch = rng.integers(0, 256, size=(n_streams, pitch), dtype=np.uint8)
        sh = C.c_int(want_shift)
        slot = L.fm_timeshift_push(ts, batch.ctypes.data, pitch, C.byref(sh), out.ctypes.data)
        for s in range(n_streams):
            r_out, r_shift, played = refs[s].push(batch[s, :CL].copy(), want_shift)
            assert (slot, sh.value) == (r_out, r_shift), (step, s)
            assert np.array_equal(out[s], played), (step, s)
            p = L.fm_timeshift_playback(ts, s)
            assert np.array_equal(np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), (CL,)), played)
        b, w, n = C.c_int(), C.c_int(), C.c_int()
        assert L.fm_timeshift_state(ts, C.byref(b), C.byref(w), C.byref(n)) == 0
        assert (b.value, w.value, n.value) == (refs[0].bottom, refs[0].full, slots)
    L.fm_timeshift_destroy(ts)


# ------------------------------------------------------------------------------------------
# the reference's own threads, offline (oracle/run_ref_player.py): harness consistency on the CPU
# ------------------------------------------------------------------------------------------
def run_ref_player(how, cap, wav, cfgname):
    import subprocess
    import sys
    c = CONFIGS[cfgname]
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_ref_player.py"), how, str(cap), str(wav),
           str(c["rate_in"]), str(c["rate_out2"]), str(c["mode"]), str(c["size"]), str(c.get("offset_tuning", 0))]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


@pytest.mark.parametrize("cfgname,kind", [("stereo192", "fm_stereo"), ("mono192", "fm_mono")])
def test_threaded_reference_pipeline_writes_the_wav_of_its_block_loop(tmp_path, cfgname, kind):
    """dongle_thread_fn + demod_thread_fn + output_thread_fn of the reference, fed by the product's file
    source through the rtlsdr_read_async contract (back-pressured on the input ring), produce exactly the
    WAV that the block loop (ref_run) + the reference's InitWaveOut/CloseWaveOut produce: nothing is lost or
    reordered in the rings, and the short tail of the capture is dropped."""
    from oracle.oracle_py import RefOracle
    ref = _ref()                                                        # the threads are the reference's own code
    blocks = 9
    iq = make_input(cfgname, kind, 3, blocks)
    cap = tmp_path / "cap.u8"
    np.concatenate([iq, np.zeros(1000, np.uint8)]).tofile(cap)          # + a short tail
    out = run_ref_player("ref", cap, tmp_path / "threads.wav", cfgname)
    assert f"{blocks} chunks delivered" in out
    pcm = RefOracle(**CONFIGS[cfgname]).run(iq)
    raw = np.ascontiguousarray(pcm).view(np.uint8)
    assert ref.ref_wav_write(str(tmp_path / "loop.wav").encode(), CONFIGS[cfgname]["mode"], raw.ctypes.data, raw.size) == 0
    assert (tmp_path / "threads.wav").read_bytes() == (tmp_path / "loop.wav").read_bytes()
