"""CPU checks of the per-stream output settings ABI (fmb_set_stream_output and friends): the entry points refuse a NULL
handle, their ctypes prototypes match the headers, the Python argument broadcasting, and the player's -e / -M flags."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from rtl_fm_player_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLAYER = os.path.join(ROOT, "rtl_fm_player_b200", "fmb_player")
NEW = ["fmb_set_stream_output", "fmb_get_stream_output", "fmb_deemph_kernel_name", "fmb_multi_set_stream_output",
       "fmb_multi_get_stream_output"]
CTYPE = {"int": C.c_int, "float *": C.POINTER(C.c_float), "double *": C.POINTER(C.c_double),
         "int *": C.POINTER(C.c_int), "char *": C.c_char_p}


def prototype(name):
    """(return type, [argument types]) of `name` as include/fmb.h or include/fmb_multi.h declares it."""
    text = "".join(open(os.path.join(ROOT, "include", f)).read() for f in ("fmb.h", "fmb_multi.h"))
    m = re.search(r"\n((?:const )?[a-z_]+ \*?)" + name + r"\(([^)]*)\);", text)
    assert m, name
    def norm(t):
        t = re.sub(r"\bconst\b", "", t).strip()
        t = re.sub(r"\s+[a-z_]+$", "", t) if not t.endswith("*") else t    # drop the parameter name
        t = re.sub(r"\s*\*\s*[a-z_]*$", " *", t).strip()
        return t
    args = [norm(a) for a in m.group(2).split(",")]
    return norm(m.group(1)), args


@pytest.mark.parametrize("name", NEW)
def test_ctypes_prototype_matches_the_header(name):
    ret, args = prototype(name)
    res, argtypes = L.SIGNATURES[name]
    assert len(args) == len(argtypes), name
    want_ret = C.c_char_p if ret == "char *" else C.c_int
    assert res is want_ret, name
    for a, t in zip(args, argtypes):
        if a in ("fmb_handle *", "fmb_multi *"):
            assert t is C.c_void_p, (name, a)
        else:
            assert t == CTYPE[a], (name, a, t)


def test_new_entry_points_refuse_a_null_handle():
    lib = R.lib()
    v = (C.c_float * 1)(1.0)
    assert lib.fmb_set_stream_output(None, 0, 1, v, None, None) == L.FMB_ERR_ARG
    assert lib.fmb_get_stream_output(None, 0, 1, v, None, None) == L.FMB_ERR_ARG
    assert lib.fmb_multi_set_stream_output(None, 0, 1, v, None, None) == L.FMB_ERR_ARG
    assert lib.fmb_multi_get_stream_output(None, 0, 1, v, None, None) == L.FMB_ERR_ARG
    assert lib.fmb_deemph_kernel_name(None) == b""


def test_python_settings_broadcast_over_the_range():
    count, args = L.stream_output_args(10, 3, 0.5, [1e-5, 0.0], None)
    assert count == 2
    assert np.array_equal(args[0][0], np.full(2, 0.5, np.float32)) and args[0][0].dtype == np.float32
    assert args[1][0].dtype == np.float64 and args[2] == (None, None)
    count, args = L.stream_output_args(10, 3, 0.5, None, 0.9)
    assert count == 7 and np.array_equal(args[2][0], np.full(7, 0.9, np.float32))
    with pytest.raises(ValueError):
        L.stream_output_args(10, 0, [1.0, 2.0], [0.0], None)


def test_player_usage_lists_the_new_flags():
    r = subprocess.run([PLAYER, "-h"], capture_output=True, text=True)
    assert "-e" in r.stderr and "-M manifest" in r.stderr and "deemph_us" in r.stderr


@pytest.mark.parametrize("line", ["cap.u8 loud", "cap.u8 0.5 -50", "cap.u8 0.5 50 extra", "cap.u8 nan",
                                  "cap.u8 0.5 inf", "cap.u8 0.4 50us"])
def test_player_refuses_a_malformed_manifest_line(tmp_path, line):
    cap = tmp_path / "cap.u8"
    cap.write_bytes(b"\x7f" * 262144)
    man = tmp_path / "channels.txt"
    man.write_text(f"# a comment\n\n{cap} 0.4 50\n{line.replace('cap.u8', str(cap))}\n")
    r = subprocess.run([PLAYER, "-M", str(man)], capture_output=True, text=True)
    assert r.returncode == 2 and "channels.txt:4" in r.stderr, r.stderr


def test_player_refuses_bad_de_emphasis_and_mixed_channel_sources(tmp_path):
    cap = tmp_path / "cap.u8"
    cap.write_bytes(b"\x7f" * 262144)
    man = tmp_path / "channels.txt"
    man.write_text(f"{cap}\n")
    for args in (["-e", "-5", str(cap)], ["-e", "x", str(cap)], ["-e", "inf", str(cap)], ["-e", "nan", str(cap)],
                 ["-M", str(man), str(cap)], ["-M", str(tmp_path / "missing.txt")]):
        r = subprocess.run([PLAYER] + args, capture_output=True, text=True)
        assert r.returncode == 2, (args, r.stderr)
    empty = tmp_path / "empty.txt"
    empty.write_text("# nothing\n")
    assert subprocess.run([PLAYER, "-M", str(empty)], capture_output=True, text=True).returncode == 2
