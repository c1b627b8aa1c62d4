"""CPU checks of the several-blocks-per-call ABI: the ctypes mirror of fmb_config ends with max_blocks_per_call, its
default means one block, and fmb_create refuses a negative maximum or a row of 2^31 bytes or more before it touches
CUDA (without a device any CUDA call would fail with FMB_ERR_CUDA instead)."""
import ctypes as C
import os
import subprocess

import pytest

import rtl_fm_player_b200 as R
from rtl_fm_player_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ctypes_mirror_ends_with_the_appended_field():
    names = [f for f, _ in L.FmbConfig._fields_]
    assert names[-2:] == ["rate_out", "max_blocks_per_call"]
    # fmb_default_config clears sizeof(fmb_config) bytes: exactly the mirror's, no more, no less
    size = C.sizeof(L.FmbConfig)
    buf = (C.c_ubyte * (size + 64))(*([0xAB] * (size + 64)))
    assert R.lib().fmb_default_config(C.cast(buf, C.POINTER(L.FmbConfig))) == 0
    cfg = L.FmbConfig.from_buffer(buf)
    assert cfg.max_blocks_per_call == 0 and cfg.block_bytes == 262144
    assert bytes(buf[size:]) == b"\xab" * 64


def test_defaults_mean_one_block_per_call():
    assert R.DemodConfig().max_blocks_per_call == 0 and R.DemodConfig().max_blocks == 1
    assert R.DemodConfig(max_blocks_per_call=8).to_c().max_blocks_per_call == 8


@pytest.mark.parametrize("block_bytes,maximum", [(262144, -1), (32768, -5), (262144, 8192), (32768, 65536),
                                                 (98304, 21846), (262144, 1 << 30)])
def test_create_refuses_a_bad_maximum_before_touching_cuda(block_bytes, maximum):
    c = L.FmbConfig()
    R.lib().fmb_default_config(C.byref(c))
    c.block_bytes, c.max_blocks_per_call = block_bytes, maximum
    h = C.c_void_p()
    assert R.lib().fmb_create(C.byref(c), C.byref(h)) == L.FMB_ERR_ARG
    assert not h.value and b"max_blocks_per_call" in R.lib().fmb_last_error()


def test_largest_accepted_maximum_gets_past_the_argument_checks():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: this would allocate 2 GB")
    c = L.FmbConfig()
    R.lib().fmb_default_config(C.byref(c))
    c.max_blocks_per_call = 8191                    # 8191 * 262144 = 2^31 - 2^18
    h = C.c_void_p()
    assert R.lib().fmb_create(C.byref(c), C.byref(h)) == L.FMB_ERR_CUDA


def test_new_entry_points_refuse_a_null_handle():
    lib = R.lib()
    assert lib.fmb_set_blocks_per_call(None, 1) == L.FMB_ERR_ARG
    assert lib.fmb_out_count_blocks(None, 1) == L.FMB_ERR_ARG
    assert lib.fmb_multi_set_blocks_per_call(None, 1) == L.FMB_ERR_ARG
    assert lib.fmb_multi_out_count_blocks(None, 1) == L.FMB_ERR_ARG


def test_player_refuses_fewer_than_one_block_per_step(tmp_path):
    player = os.path.join(ROOT, "rtl_fm_player_b200", "fmb_player")
    cap = tmp_path / "x.u8"
    cap.write_bytes(b"\x7f" * 262144)
    r = subprocess.run([player, "-K", "0", str(cap)], capture_output=True, text=True)
    assert r.returncode == 2 and "-K" in r.stderr
    r = subprocess.run([player, "-h"], capture_output=True, text=True)
    assert "-K" in r.stderr
