"""The fused restatement (oracle/fm_oracle.c built with FMO_FMA, PortOracle(fma=True)) is the definition of
FMB_PRECISION_FMA: the FIR multiply-adds fused with fmaf, in the reference's order, everything else rounded as in the
reference.  These CPU tests pin the model itself, so that on the GPU the FMA kernels only have to equal it bit for bit
(tests/test_gpu_fma.py):

  * it is within +-1 LSB of int16 PCM of the reference's own output on every golden case and the three 10 s captures
    (the tolerance the FMA mode documents);
  * it really fuses: on programme material its PCM and its discriminator output differ from the exact build's;
  * its carried state resumes bit-exactly across block boundaries.
"""
import json
import os

import numpy as np
import pytest

from oracle.oracle_py import PortOracle
from vectors import B, CASES, CONFIGS, LONG_CASES, long_capture_bytes, make_input, sha

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "golden.npz"))
META = json.load(open(os.path.join(HERE, "golden", "golden_meta.json")))

PROGRAMME = ("fm_stereo", "fm_mono", "random")       # synth kinds with signal in every FIR tap
_BASE = ["tb", "pre_r", "pre_j", "br", "deemph_l"]
CARRIED = {0: _BASE, 1: _BASE, 2: _BASE + ["bm", "bs", "pp", "deemph_r"]}   # the state each decoder mode carries


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def max_lsb(a, b):
    assert a.shape == b.shape
    return int(np.abs(a.astype(np.int32) - b.astype(np.int32)).max(initial=0))


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_fused_restatement_is_within_one_lsb_of_the_reference(case):
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    assert sha(iq) == META["cases"][cid]["input_sha256"]
    got = PortOracle(**CONFIGS[cfg], fma=True).run(iq)
    assert max_lsb(got, GOLD[cid]) <= 1


@pytest.mark.parametrize("case", LONG_CASES, ids=[c[0] for c in LONG_CASES])
def test_fused_restatement_long_captures_within_one_lsb(case):
    """The golden data of the 10 s captures is a hash: the exact build is checked against it, then the fused build
    against the exact one."""
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    iq = np.concatenate([iq, np.zeros(long_capture_bytes(cfg) - blocks * B, np.uint8)])
    exact = PortOracle(**CONFIGS[cfg]).run(iq)
    assert sha(exact) == META["long"][cid]["pcm_sha256"]
    fused = PortOracle(**CONFIGS[cfg], fma=True).run(iq)
    assert max_lsb(fused, exact) <= 1
    print(f"\n{cid}: {int((fused != exact).sum())} of {fused.size} PCM samples differ by 1 LSB")


@pytest.mark.parametrize("case", [c for c in CASES if c[2] in PROGRAMME], ids=[c[0] for c in CASES if c[2] in PROGRAMME])
def test_fused_build_really_fuses(case):
    """A fused build that silently compiled to the exact form would pass the +-1 LSB test; it cannot pass this one.
    Every programme-material case differs from the exact build in the discriminator output (the channel FIR) and in the
    decoder output of its first block, and somewhere in its PCM."""
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    fo, eo = PortOracle(**CONFIGS[cfg], fma=True), PortOracle(**CONFIGS[cfg])
    _, fs = fo.block(iq[:B], stages=True)
    _, es = eo.block(iq[:B], stages=True)
    assert not np.array_equal(bits(fs["dem"]), bits(es["dem"])), "discriminator output is the exact build's"
    assert not np.array_equal(bits(fs["lr"]), bits(es["lr"])), "decoder output is the exact build's"
    fused, exact = PortOracle(**CONFIGS[cfg], fma=True).run(iq), GOLD[cid]
    assert (fused != exact).any(), "PCM is the exact build's"


@pytest.mark.parametrize("cfg,kind", [("stereo240", "fm_stereo"), ("stereo170_44", "random"), ("mono240_32", "fm_mono"),
                                      ("mono192", "random"), ("drop192", "fm_stereo")])
def test_fused_state_round_trip(cfg, kind):
    """fmo_get_state / fmo_set_state: a fresh fused oracle that takes over the carried state and resampler phase at
    every block boundary continues bit-exactly, every stage, as one that ran the whole capture."""
    blocks = 5
    iq = make_input(cfg, kind, 3, blocks)
    whole = PortOracle(**CONFIGS[cfg], fma=True)
    prev = None
    for b in range(blocks):
        blk = iq[b * B:(b + 1) * B]
        o = PortOracle(**CONFIGS[cfg], fma=True)
        if prev is not None:
            o.set_state(*prev.state())
        p_whole, s_whole = whole.block(blk, stages=True)
        p_o, s_o = o.block(blk, stages=True)
        assert np.array_equal(p_o, p_whole), f"block {b}: PCM"
        for k in ("dem", "lr", "de"):
            assert np.array_equal(bits(s_o[k]), bits(s_whole[k])), f"block {b}: stage {k}"
        (so, *so_pos), (sw, *sw_pos) = o.state(), whole.state()
        assert so_pos == sw_pos, f"block {b}: phase / blocks done"
        for f in CARRIED[CONFIGS[cfg]["mode"]]:     # mono never writes bm / bs (their bytes are scratch)
            a, w = (np.array(getattr(x, f), dtype=np.float32, ndmin=1) for x in (so, sw))
            assert np.array_equal(bits(a), bits(w)), f"block {b}: carried {f}"
        prev = o
