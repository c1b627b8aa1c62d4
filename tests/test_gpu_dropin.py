"""GPU parity of the drop-in entry points (include/fm_dropin.h) and of the offline batch player.

The struct handed to our full_demod() is a `struct demod_state` in the reference's own layout
(csrc/ref_layout.h).  Every test runs against the C restatement (oracle/fm_oracle.c), whose PCM and
filter tables tests/golden pins bit for bit to the reference's; the struct is then set up the way
oracle/ref_harness.c:ref_create sets the fields full_demod reads.  Where the reference itself is built
(oracle/_ref/libfmref.so), each test also runs against it: the struct is then the reference's own,
allocated and initialised by its demod_init + init_lp_real_f32 (src/rtl_fm_player.c:1156, :413), and a
twin struct runs the reference's CPU functions on the same bytes.
Bar: int16 PCM and every carried state field bit-identical."""
import ctypes as C
import functools
import math
import os
import subprocess

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from oracle.oracle_py import REF_CLI, REF_PATH, PortOracle, PortState, ref_available
from vectors import B, CONFIGS, make_input

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = np.load(os.path.join(HERE, "golden", "golden.npz"))


def layout():
    out = {}
    for line in open(os.path.join(ROOT, "rtl_fm_player_b200", "csrc", "ref_layout.h")):
        f = line.split()
        if len(f) == 3 and f[0] == "#define" and f[2].isdigit():
            out[f[1]] = int(f[2])
    return out


LAY = layout()


@pytest.fixture(scope="module")
def ours():
    lib = C.CDLL(R.LIB_PATH)
    for n in ("rotate_90_u8_f32", "u8_f32", "full_demod", "fm_dropin_release", "init_lp_real_f32", "deinit_lp_real_f32"):
        getattr(lib, n).argtypes = [C.c_void_p]
        getattr(lib, n).restype = None
    for n in ("fm_dropin_export_state", "fm_dropin_import_state"):
        getattr(lib, n).argtypes = [C.c_void_p]
    return lib


def field(d, off, ctype):
    return ctype.from_address(d + off)


def lpr(d, name, ctype):
    return field(d, LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_" + name], ctype)


def ours_block(ours, d, iq, offset_tuning):
    """What demod_thread_fn does with one chunk (:870-889), calling OUR symbols on the struct."""
    C.memmove(d + LAY["FMD_OFF_buf"], iq.ctypes.data, iq.size)
    field(d, LAY["FMD_OFF_buf_len"], C.c_uint32).value = iq.size
    (ours.u8_f32 if offset_tuning else ours.rotate_90_u8_f32)(d)
    assert field(d, LAY["FMD_OFF_lp_len"], C.c_int).value == iq.size
    ours.full_demod(d)
    n = field(d, LAY["FMD_OFF_result_len"], C.c_int).value
    return np.frombuffer((C.c_char * (2 * n)).from_address(d + LAY["FMD_OFF_result"]), dtype=np.int16).copy()


# ------------------------------------------------------------------------------------------
# against the C restatement: the struct set up by the test, our init_lp_real_f32 for its arrays
# ------------------------------------------------------------------------------------------
class Struct:
    """A struct demod_state with the fields full_demod reads set as ref_create sets them (the numerics flags,
    deemph_lambda as main computes it, :1575-1578) and the decoder arrays of OUR init_lp_real_f32 (pinned to the
    reference's tables by test_our_init_lp_real_f32_fills_the_struct_like_the_reference).  Every other field is
    zero; our entry points read none of them."""

    def __init__(self, ours, cfgname, **over):
        kw = dict(CONFIGS[cfgname]); kw.update(over)
        self.ours, self.kw = ours, kw
        self.buf = C.create_string_buffer(LAY["FMD_SIZEOF_DEMOD_STATE"])
        d = self.d = C.addressof(self.buf)
        rate_out = kw.get("rate_out") or kw["rate_in"]
        deemph, volume = kw.get("deemph", 0.000050), kw.get("volume", 0.4)
        for name, v in (("rate_in", kw["rate_in"]), ("rate_out", rate_out), ("rate_out2", kw["rate_out2"]),
                        ("offset_tuning", kw.get("offset_tuning", 0))):
            field(d, LAY["FMD_OFF_" + name], C.c_int).value = v
        lpr(d, "mode", C.c_int).value = kw["mode"]
        lpr(d, "size", C.c_int).value = kw["size"]
        field(d, LAY["FMD_OFF_deemph"], C.c_double).value = deemph
        field(d, LAY["FMD_OFF_volume"], C.c_float).value = volume
        if deemph:
            output_rate = kw["rate_out2"] or rate_out
            field(d, LAY["FMD_OFF_deemph_lambda"], C.c_float).value = math.exp(-1.0 / (output_rate * deemph))
        ours.init_lp_real_f32(d)

    def block(self, iq):
        return ours_block(self.ours, self.d, iq, self.kw.get("offset_tuning", 0))

    def close(self):
        self.ours.deinit_lp_real_f32(self.d)                         # releases the GPU context too


def twin(cfgname, **over):
    kw = dict(CONFIGS[cfgname]); kw.update(over)
    return PortOracle(**kw)


def rings(kw):
    """The decoder rings the reference carries between blocks: br when lpr runs (rate_out2 > 0, mode >= 1),
    bm and bs in stereo."""
    if kw["rate_out2"] <= 0 or kw["mode"] < 1:
        return ()
    return ("br", "bm", "bs") if kw["mode"] == 2 else ("br",)


def ring_pos(kw, blocks):
    """lpr.pos after `blocks` whole blocks: lp_real_f32 writes one ring slot per demodulated sample (buf_len / 16
    of them a block, :500-566) wherever it runs; elsewhere pos stays where init_lp_real_f32 put it."""
    return blocks * (B // 16) % kw["size"] if rings(kw) else 0


def f32(*xs):
    return np.array(xs, np.float32).tobytes()


def struct_state(s):
    """Every carried field of the struct, in the reference's own representation (raw rings, pos)."""
    d, size = s.d, s.kw["size"]
    out = {
        "lowpass_tb": bytes((C.c_char * 192).from_address(d + LAY["FMD_OFF_lowpass_tb"])),
        "pre": bytes((C.c_char * 8).from_address(d + LAY["FMD_OFF_pre_r_f32"])),
        "deemph": bytes((C.c_char * 8).from_address(d + LAY["FMD_OFF_deemph_l_f32"])),
        "prev_lpr_index": field(d, LAY["FMD_OFF_prev_lpr_index"], C.c_int).value,
        "pos": lpr(d, "pos", C.c_int).value,
        "pp": bytes((C.c_char * 4).from_address(d + LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_pp"])),
    }
    for ring in rings(s.kw):
        out[ring] = bytes((C.c_char * (4 * size)).from_address(lpr(d, ring, C.c_void_p).value))
    return out


def twin_state(port, kw, blocks):
    """The same fields as the reference would hold them after `blocks` blocks: the restatement keeps each ring as a
    history, oldest to newest, at the end of 128 floats; the reference's ring holds the oldest at pos."""
    st, phase, _ = port.state()
    pos = ring_pos(kw, blocks)
    out = {"lowpass_tb": f32(*st.tb), "pre": f32(st.pre_r, st.pre_j), "deemph": f32(st.deemph_l, st.deemph_r),
           "prev_lpr_index": phase, "pos": pos, "pp": f32(st.pp)}
    for ring in rings(kw):
        out[ring] = np.roll(np.frombuffer(f32(*getattr(st, ring))[-4 * kw["size"]:], np.float32), pos).tobytes()
    return out


def write_twin_state(s, port, blocks):
    """The CPU side hands over: its carried fields written into the struct as the reference would leave them."""
    d, kw = s.d, s.kw
    want = twin_state(port, kw, blocks)
    C.memmove(d + LAY["FMD_OFF_lowpass_tb"], want["lowpass_tb"], 192)
    C.memmove(d + LAY["FMD_OFF_pre_r_f32"], want["pre"], 8)
    C.memmove(d + LAY["FMD_OFF_deemph_l_f32"], want["deemph"], 8)
    field(d, LAY["FMD_OFF_prev_lpr_index"], C.c_int).value = want["prev_lpr_index"]
    lpr(d, "pos", C.c_int).value = want["pos"]
    C.memmove(d + LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_pp"], want["pp"], 4)
    for ring in rings(kw):
        C.memmove(lpr(d, ring, C.c_void_p).value, want[ring], 4 * kw["size"])


def twin_from_struct(s, blocks):
    """A CPU twin that starts from nothing but the struct: the restatement given the struct's carried fields."""
    d, kw = s.d, s.kw
    st = PortState()
    st.tb[:] = np.frombuffer(bytes((C.c_char * 192).from_address(d + LAY["FMD_OFF_lowpass_tb"])), np.float32).tolist()
    st.pre_r, st.pre_j = (field(d, LAY[n], C.c_float).value for n in ("FMD_OFF_pre_r_f32", "FMD_OFF_pre_j_f32"))
    st.deemph_l, st.deemph_r = (field(d, LAY[n], C.c_float).value for n in ("FMD_OFF_deemph_l_f32", "FMD_OFF_deemph_r_f32"))
    st.pp = lpr(d, "pp", C.c_float).value
    size, pos = kw["size"], lpr(d, "pos", C.c_int).value
    for ring in rings(kw):
        hist = np.zeros(128, np.float32)
        hist[-size:] = np.roll(np.frombuffer(bytes((C.c_char * (4 * size)).from_address(lpr(d, ring, C.c_void_p).value)),
                                             np.float32), -pos)
        getattr(st, ring)[:] = hist.tolist()
    port = PortOracle(**kw)
    port.set_state(st, field(d, LAY["FMD_OFF_prev_lpr_index"], C.c_int).value, blocks)
    return port


# ------------------------------------------------------------------------------------------
# against the reference itself, where oracle/_ref/libfmref.so is built
# ------------------------------------------------------------------------------------------
class RefCfg(C.Structure):
    _fields_ = [("rate_in", C.c_int), ("rate_out2", C.c_int), ("mode", C.c_int), ("size", C.c_int),
                ("offset_tuning", C.c_int), ("deemph", C.c_double), ("volume", C.c_float), ("rate_out", C.c_int)]


@functools.cache
def ref_lib():
    ref = C.CDLL(REF_PATH)
    ref.ref_create.restype = C.c_void_p
    ref.ref_create.argtypes = [C.POINTER(RefCfg)]
    ref.ref_destroy.argtypes = [C.c_void_p]
    ref.ref_demod_state.restype = C.c_void_p
    ref.ref_demod_state.argtypes = [C.c_void_p]
    ref.ref_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    ref.ref_wav_write.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_size_t]
    return ref


def new_ref(ref, cfgname, **over):
    kw = dict(CONFIGS[cfgname]); kw.update(over)
    c = RefCfg(kw["rate_in"], kw["rate_out2"], kw["mode"], kw["size"], kw.get("offset_tuning", 0),
               kw.get("deemph", 0.000050), kw.get("volume", 0.4), kw.get("rate_out", 0))
    h = ref.ref_create(C.byref(c))
    assert h
    return h, ref.ref_demod_state(h)


def state_bytes(d, mode):
    """Every carried field of the reference struct, in the reference's own representation."""
    size = field(d, LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_size"], C.c_int).value
    out = {
        "lowpass_tb": bytes((C.c_char * 192).from_address(d + LAY["FMD_OFF_lowpass_tb"])),
        "pre": bytes((C.c_char * 8).from_address(d + LAY["FMD_OFF_pre_r_f32"])),
        "deemph": bytes((C.c_char * 8).from_address(d + LAY["FMD_OFF_deemph_l_f32"])),
        "prev_lpr_index": field(d, LAY["FMD_OFF_prev_lpr_index"], C.c_int).value,
        "pos": field(d, LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_pos"], C.c_int).value,
        "pp": bytes((C.c_char * 4).from_address(d + LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_pp"])),
    }
    for ring in ("br",) + (("bm", "bs") if mode == 2 else ()):
        ptr = field(d, LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_" + ring], C.c_void_p).value
        out[ring] = bytes((C.c_char * (4 * size)).from_address(ptr))
    return out


def ref_block(ref, h, iq):
    pcm = np.empty(131072, np.int16)
    n = ref.ref_block(h, iq.ctypes.data, iq.size, pcm.ctypes.data)
    return pcm[:n].copy()


def full_demod_against_the_reference(ours, cfgname, kind):
    ref = ref_lib()
    kw = CONFIGS[cfgname]
    off, mode = kw.get("offset_tuning", 0), kw["mode"]
    blocks = 7
    iq = make_input(cfgname, kind, 11, blocks)
    h_ref, d_ref = new_ref(ref, cfgname)          # runs the reference's CPU code
    h_gpu, d_gpu = new_ref(ref, cfgname)          # same struct type, demodulated by libfmb.so
    try:
        for b in range(4):
            blk = iq[b * B:(b + 1) * B]
            assert np.array_equal(ours_block(ours, d_gpu, blk, off), ref_block(ref, h_ref, blk)), f"block {b}"
        # GPU state -> struct: every carried field equals the reference's, in its own representation
        assert ours.fm_dropin_export_state(d_gpu) == 0
        assert state_bytes(d_gpu, mode) == state_bytes(d_ref, mode)
        # ... so the REFERENCE can carry on from the exported struct (GPU -> CPU hand-over)
        ours.fm_dropin_release(d_gpu)
        blk = iq[4 * B:5 * B]
        assert np.array_equal(ref_block(ref, h_gpu, blk), ref_block(ref, h_ref, blk))
        # ... and the GPU can carry on from a struct the reference advanced (CPU -> GPU hand-over)
        for b in (5, 6):
            blk = iq[b * B:(b + 1) * B]
            assert np.array_equal(ours_block(ours, d_gpu, blk, off), ref_block(ref, h_ref, blk)), f"block {b}"
        assert ours.fm_dropin_export_state(d_gpu) == 0
        assert state_bytes(d_gpu, mode) == state_bytes(d_ref, mode)
    finally:
        ours.fm_dropin_release(d_gpu)
        ref.ref_destroy(h_ref)
        ref.ref_destroy(h_gpu)


def init_again_against_the_reference(ours):
    ref = ref_lib()
    iq = make_input("stereo192", "random", 5, 2)
    h_ref, d_ref = new_ref(ref, "stereo192")
    h_gpu, d_gpu = new_ref(ref, "stereo192")
    try:
        blk = iq[:B]
        assert np.array_equal(ours_block(ours, d_gpu, blk, 0), ref_block(ref, h_ref, blk))
        # both sides re-init WITHOUT deinit (leaks the old rings, as the reference would): rings zeroed, pos 0,
        # pp 0, everything else (lowpass_tb, pre_*, de-emphasis, resampler phase) carried on
        ours.init_lp_real_f32(d_gpu)
        ref2 = C.CDLL(REF_PATH)
        if not hasattr(ref2, "ref_init_lp_real"):
            pytest.skip("reference harness without the re-init hook")
        ref2.ref_init_lp_real.argtypes = [C.c_void_p]
        ref2.ref_init_lp_real(h_ref)
        blk = iq[B:2 * B]
        assert np.array_equal(ours_block(ours, d_gpu, blk, 0), ref_block(ref, h_ref, blk))
    finally:
        ours.fm_dropin_release(d_gpu)
        ref.ref_destroy(h_ref)
        ref.ref_destroy(h_gpu)


def volume_change_against_the_reference(ours):
    ref = ref_lib()
    iq = make_input("stereo192", "random", 3, 3)
    h_ref, d_ref = new_ref(ref, "stereo192")
    h_gpu, d_gpu = new_ref(ref, "stereo192")
    ours.fm_dropin_set_strict(1)
    try:
        for b, vol in enumerate((0.4, 1.0, 0.05)):                      # the player's volume keys change demod.volume
            for d in (d_ref, d_gpu):
                field(d, LAY["FMD_OFF_volume"], C.c_float).value = vol
            blk = iq[b * B:(b + 1) * B]
            assert np.array_equal(ours_block(ours, d_gpu, blk, 0), ref_block(ref, h_ref, blk))
            assert state_bytes(d_gpu, 2) == state_bytes(d_ref, 2)       # strict: struct current after every call
    finally:
        ours.fm_dropin_set_strict(0)
        ours.fm_dropin_release(d_gpu)
        ref.ref_destroy(h_ref)
        ref.ref_destroy(h_gpu)


def our_init_against_the_reference(ours):
    ref = ref_lib()
    h_ref, d_ref = new_ref(ref, "stereo240")
    h_x, d_x = new_ref(ref, "stereo240")
    try:
        ours.deinit_lp_real_f32(d_x)                                     # frees the reference's arrays (:455-470)
        assert field(d_x, LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_rsize"], C.c_int).value == 0
        ours.init_lp_real_f32(d_x)                                       # ours: allocate + design
        for name in ("fm", "fp", "fs"):
            pa = field(d_ref, LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_" + name], C.c_void_p).value
            pb = field(d_x, LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_" + name], C.c_void_p).value
            assert bytes((C.c_char * 180).from_address(pa)) == bytes((C.c_char * 180).from_address(pb)), name
        lo, hi = LAY["FMD_OFF_lpr"] + LAY["FMD_LPR_OFF_swf"], LAY["FMD_OFF_lpr"] + LAY["FMD_SIZEOF_LP_REAL"]
        assert bytes((C.c_char * (hi - lo)).from_address(d_ref + lo)) == bytes((C.c_char * (hi - lo)).from_address(d_x + lo))
        iq = make_input("stereo240", "fm_stereo", 1, 2)
        for b in range(2):
            blk = iq[b * B:(b + 1) * B]
            assert np.array_equal(ours_block(ours, d_x, blk, 0), ref_block(ref, h_ref, blk))
    finally:
        ours.fm_dropin_release(d_x)
        ref.ref_destroy(h_ref)
        ref.ref_destroy(h_x)


# ------------------------------------------------------------------------------------------
# the tests
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfgname,kind", [("stereo192", "fm_stereo"), ("stereo240", "random"), ("mono192", "fm_mono"),
                                          ("stereo192_off", "random"), ("mono240_off", "fm_mono"), ("drop192", "fm_stereo"),
                                          ("nolpr192", "random"), ("nodeemph192", "random"),
                                          # -o 2: the struct has rate_in = 2*rate_out (main :1510); lp_real_f32 ticks
                                          # at rate_out (:485) while the filters follow rate_in
                                          ("stereo384_o2", "fm_stereo"), ("stereo480_o2", "random")])
def test_full_demod_on_the_references_struct_is_bit_identical(ours, cfgname, kind):
    blocks = 7
    iq = make_input(cfgname, kind, 11, blocks)
    blk = [iq[b * B:(b + 1) * B] for b in range(blocks)]
    s, port = Struct(ours, cfgname), twin(cfgname)
    try:
        for b in range(4):
            assert np.array_equal(s.block(blk[b]), port.block(blk[b])), f"block {b}"
        # GPU state -> struct: every carried field as the reference holds it
        assert ours.fm_dropin_export_state(s.d) == 0
        assert struct_state(s) == twin_state(port, s.kw, 4)
        # ... so the CPU can carry on from the exported struct alone (GPU -> CPU hand-over)
        ours.fm_dropin_release(s.d)
        cpu = twin_from_struct(s, 4)
        assert np.array_equal(cpu.block(blk[4]), port.block(blk[4])), "block 4"
        # ... and the GPU can carry on from a struct the CPU advanced (CPU -> GPU hand-over)
        write_twin_state(s, cpu, 5)
        for b in (5, 6):
            assert np.array_equal(s.block(blk[b]), port.block(blk[b])), f"block {b}"
        assert ours.fm_dropin_export_state(s.d) == 0
        assert struct_state(s) == twin_state(port, s.kw, 7)
    finally:
        s.close()
    if ref_available():
        full_demod_against_the_reference(ours, cfgname, kind)


def test_init_lp_real_f32_again_restarts_the_gpu_history(ours):
    """The reference's init_lp_real_f32 callocs fresh rings (:430-436); called again on a struct that already has
    a GPU context, ours must forget the GPU copy of the history too."""
    iq = make_input("stereo192", "random", 5, 2)
    s, port = Struct(ours, "stereo192"), twin("stereo192")
    try:
        blk = iq[:B]
        assert np.array_equal(s.block(blk), port.block(blk))
        # re-init WITHOUT deinit (leaks the old rings, as the reference would): rings zeroed, pos 0, pp 0,
        # everything else (lowpass_tb, pre_*, de-emphasis, resampler phase) carried on
        ours.init_lp_real_f32(s.d)
        st, phase, done = port.state()
        for ring in ("br", "bm", "bs"):
            setattr(st, ring, (C.c_float * 128)())
        st.pp = 0.0
        port.set_state(st, phase, done)
        blk = iq[B:2 * B]
        assert np.array_equal(s.block(blk), port.block(blk))
    finally:
        s.close()
    if ref_available():
        init_again_against_the_reference(ours)


def test_volume_change_and_strict_mode(ours):
    iq = make_input("stereo192", "random", 3, 3)
    s = Struct(ours, "stereo192")
    port = None
    ours.fm_dropin_set_strict(1)
    try:
        for b, vol in enumerate((0.4, 1.0, 0.05)):                      # the player's volume keys change demod.volume
            field(s.d, LAY["FMD_OFF_volume"], C.c_float).value = vol
            nxt = twin("stereo192", volume=vol)                         # the twin carries its state over to the new volume
            if port is not None:
                nxt.set_state(*port.state())
            port = nxt
            blk = iq[b * B:(b + 1) * B]
            assert np.array_equal(s.block(blk), port.block(blk))
            assert struct_state(s) == twin_state(port, s.kw, b + 1)    # strict: struct current after every call
    finally:
        ours.fm_dropin_set_strict(0)
        s.close()
    if ref_available():
        volume_change_against_the_reference(ours)


def test_our_init_lp_real_f32_fills_the_struct_like_the_reference(ours):
    s = Struct(ours, "stereo240")
    try:
        ours.deinit_lp_real_f32(s.d)                                     # frees the arrays (:455-470)
        assert lpr(s.d, "rsize", C.c_int).value == 0
        ours.init_lp_real_f32(s.d)                                       # ours: allocate + design
        for name in ("fm", "fp", "fs"):                                  # the reference's own tables (tests/golden)
            got = np.frombuffer(bytes((C.c_char * 180).from_address(lpr(s.d, name, C.c_void_p).value)), np.float32)
            assert got.tobytes() == GOLD[f"tab_240k_90_{name}"].astype(np.float32).tobytes(), name
        misc = GOLD["tab_240k_90_misc"].astype(np.float32)
        assert f32(lpr(s.d, "swf", C.c_float).value, lpr(s.d, "cwf", C.c_float).value) == misc[:2].tobytes()
        assert lpr(s.d, "pp", C.c_float).value == 0.0 and lpr(s.d, "pos", C.c_int).value == 0
        assert (lpr(s.d, "size", C.c_int).value, lpr(s.d, "rsize", C.c_int).value, lpr(s.d, "mode", C.c_int).value) == (90, 45, 2)
        iq = make_input("stereo240", "fm_stereo", 1, 2)
        port = twin("stereo240")
        for b in range(2):
            blk = iq[b * B:(b + 1) * B]
            assert np.array_equal(s.block(blk), port.block(blk))
    finally:
        s.close()
    if ref_available():
        our_init_against_the_reference(ours)


def wav_of(pcm, mode, path):
    """The WAV file include/fm_wav.h writes for this PCM.  Its header is pinned to the reference's by a stored hash
    (tests/test_host_c.py::test_wav_header_is_the_references), the whole file to the reference's writer only where
    oracle/_ref is built; so the reference leg of test_fmb_player_wav_files_equal_the_reference_pipeline frames the
    expected PCM with the reference's own writer."""
    L = C.CDLL(R.LIB_PATH)
    L.fm_wav_open.argtypes = [C.POINTER(C.c_void_p), C.c_char_p, C.c_int]
    L.fm_wav_write.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.fm_wav_close.argtypes = [C.c_void_p]
    raw = np.ascontiguousarray(pcm).view(np.uint8)
    w = C.c_void_p()
    assert L.fm_wav_open(C.byref(w), str(path).encode(), mode) == 0
    assert L.fm_wav_write(w, raw.ctypes.data, raw.size) == 0
    assert L.fm_wav_close(w) == 0
    return open(path, "rb").read()


@pytest.mark.parametrize("flag,cfgname,kind", [("-X", "stereo192", "fm_stereo"), ("-Y", "mono192", "fm_mono")])
def test_fmb_player_wav_files_equal_the_reference_pipeline(tmp_path, flag, cfgname, kind):
    """BASELINE configs[0]/[1] end to end in C: capture files -> fmb_player (file source, CUDA, WAV writer) vs
    the block loop of the C restatement over the same files (whole blocks; the tail is never demodulated) and,
    where it is built, the reference's own code (ref_offline PCM -> the reference's InitWaveOut/CloseWaveOut)."""
    player = os.path.join(ROOT, "rtl_fm_player_b200", "fmb_player")
    mode = CONFIGS[cfgname]["mode"]
    lens = [9, 12, 5]                                                   # channels of different lengths (blocks) + a tail
    files, want = [], []
    for s, nb in enumerate(lens):
        p = tmp_path / f"ch{s}.u8"
        cap = np.concatenate([make_input(cfgname, kind, s, nb), np.full(1000 * (s + 1), 127, np.uint8)])
        cap.tofile(p)
        files.append(str(p))
        want.append(PortOracle(**CONFIGS[cfgname]).run(cap))
    r = subprocess.run([player, flag, "-w", *files], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    for s, f in enumerate(files):
        assert open(f + ".wav", "rb").read() == wav_of(want[s], mode, tmp_path / f"want{s}.wav"), f"channel {s}"
        if os.path.exists(REF_CLI):
            pcm_path = tmp_path / f"ref{s}.pcm"
            subprocess.run([REF_CLI, flag, f, str(pcm_path)], check=True, capture_output=True)
            pcm = np.fromfile(pcm_path, dtype=np.uint8)
            theirs = tmp_path / f"ref{s}.wav"
            assert ref_lib().ref_wav_write(str(theirs).encode(), mode, pcm.ctypes.data, pcm.size) == 0
            assert open(f + ".wav", "rb").read() == theirs.read_bytes(), f"channel {s}"
    # the same channels sharded over several devices by the C multi-GPU host (-d: every visible GPU, or three shards
    # sharing GPU 0 on a 1-GPU box): byte-identical WAV files again
    ndev = R.device_count()
    dlist = f"0-{ndev - 1}" if ndev >= 2 else "0,0,0"
    for f in files:
        os.rename(f + ".wav", f + ".single.wav")
    r = subprocess.run([player, flag, "-w", "-d", dlist, *files], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert f"on {min(max(ndev, 3) if ndev < 2 else ndev, len(files))} device(s)" in r.stderr, r.stderr
    for f in files:
        assert open(f + ".wav", "rb").read() == open(f + ".single.wav", "rb").read(), f
    # raw PCM output keeps every sample (no cluster rule)
    r = subprocess.run([player, flag, files[0]], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(files[0] + ".pcm", "rb").read() == want[0].tobytes()
    if os.path.exists(REF_CLI):
        subprocess.run([REF_CLI, flag, files[0], str(tmp_path / "r.pcm")], check=True, capture_output=True)
        assert open(files[0] + ".pcm", "rb").read() == (tmp_path / "r.pcm").read_bytes()


@pytest.mark.parametrize("cfgname,kind,blocks", [("stereo192", "fm_stereo", 9), ("stereo240", "random", 13),
                                                 ("mono192", "fm_mono", 9), ("stereo192_off", "fm_stereo", 9)])
def test_unmodified_player_threads_with_libfmb_interposed_write_the_same_wav(tmp_path, cfgname, kind, blocks):
    """The strongest form of the drop-in claim: the reference's OWN dongle/demod/output threads (compiled
    unmodified into oracle/_ref/libfmref.so) run a capture file twice in separate processes -- once bound to
    the reference's CPU functions, once with rtl_fm_player_b200/libfmb.so first in the global symbol scope
    (what LD_PRELOAD does for the real binary), so that their calls to init_*/rotate_90_u8_f32/u8_f32/
    full_demod land in the CUDA drop-in.  The two WAV files must be byte-identical."""
    import sys
    if not os.path.exists(REF_PATH):
        pytest.skip("oracle/_ref/libfmref.so missing")
    c = CONFIGS[cfgname]
    iq = make_input(cfgname, kind, 5, blocks)
    cap = tmp_path / "cap.u8"
    iq.tofile(cap)
    outs = {}
    for how in ("ref", "dropin"):
        wav = tmp_path / f"{how}.wav"
        cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_ref_player.py"), how, str(cap), str(wav),
               str(c["rate_in"]), str(c["rate_out2"]), str(c["mode"]), str(c["size"]), str(c.get("offset_tuning", 0))]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and f"{blocks} chunks delivered" in r.stdout, r.stdout + r.stderr
        outs[how] = wav.read_bytes()
    assert len(outs["ref"]) > 260 + 32768
    assert outs["dropin"] == outs["ref"]
