"""The CPU oracle is pinned here (CPU-only tests).

  * against the reference's OWN code compiled unmodified (oracle/_ref/libfmref.so), every stage,
    bit for bit -- runs wherever that build exists (the build container; the prebuilt .so also
    travels to the GPU box);
  * against tests/golden/golden.npz, PCM that the reference build produced (made by
    tests/golden/make_golden.py), so the pin holds where the reference is absent.
"""
import json
import os

import numpy as np
import pytest

from oracle.oracle_py import PortOracle, RefOracle, ref_available
from vectors import B, CASE_BY_ID, CASES, CONFIGS, LONG_CASES, long_capture_bytes, make_input, sha

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "golden.npz"))
META = json.load(open(os.path.join(HERE, "golden", "golden_meta.json")))


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_port_matches_golden_pcm(case):
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    assert sha(iq) == META["cases"][cid]["input_sha256"], "synthetic generator no longer reproduces the golden input bytes"
    port = PortOracle(**CONFIGS[cfg])
    got = np.concatenate([port.block(iq[b * B:(b + 1) * B]) for b in range(blocks)])
    assert got.dtype == np.int16
    assert np.array_equal(got, GOLD[cid]), "port oracle PCM differs from the reference's PCM (bit-exact required)"


@pytest.mark.skipif(not ref_available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_port_matches_reference_every_stage(case):
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    ref, port = RefOracle(**CONFIGS[cfg]), PortOracle(**CONFIGS[cfg])
    for b in range(blocks):
        p_ref, s_ref = ref.block(iq[b * B:(b + 1) * B], stages=True)
        p_port, s_port = port.block(iq[b * B:(b + 1) * B], stages=True)
        for k in ("dem", "lr", "de"):
            assert np.array_equal(bits(s_ref[k]), bits(s_port[k])), f"block {b}: stage {k} differs"
        assert np.array_equal(p_ref, p_port), f"block {b}: PCM differs"


@pytest.mark.skipif(not ref_available(), reason="oracle/_ref not built")
def test_reference_stage_calls_equal_full_demod():
    """ref_block_stages (stage functions called one by one) == full_demod (:758-788)."""
    iq = make_input("stereo240", "random", 3, 3)
    a, b = RefOracle(**CONFIGS["stereo240"]), RefOracle(**CONFIGS["stereo240"])
    for k in range(3):
        assert np.array_equal(a.block(iq[k * B:(k + 1) * B]), b.block(iq[k * B:(k + 1) * B], stages=True)[0])


@pytest.mark.parametrize("case", LONG_CASES, ids=[c[0] for c in LONG_CASES])
def test_port_long_capture_configs_0_and_1(case):
    """BASELINE.json configs[0]/[1]: 10 s single-channel captures, 117 full blocks at 8 x 192 kHz; configs[0] also at
    the literal default rate (8 x 240 kHz, rotate path): 146 full blocks."""
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    m = META["long"][cid]
    assert sha(iq) == m["input_sha256"]
    pcm = PortOracle(**CONFIGS[cfg]).run(np.concatenate([iq, np.zeros(long_capture_bytes(cfg) - blocks * B, np.uint8)]))
    assert pcm.size == m["n_pcm"]          # the tail short of a block (49 152 B at 192 k) is dropped (:863-868)
    assert sha(pcm) == m["pcm_sha256"]


@pytest.mark.parametrize("name", ["192k_90", "192k_128", "240k_90", "240k_128"])
def test_port_filter_tables_match_reference(name):
    kw = META["tables"][name]
    t = PortOracle(mode=2, **kw).tables()
    for k in ("fb", "fm", "fp", "fs"):
        assert np.array_equal(bits(t[k]), bits(GOLD[f"tab_{name}_{k}"])), k
    assert np.array_equal(bits(t["misc"][:3]), bits(GOLD[f"tab_{name}_misc"]))  # swf, cwf, lambda


def test_known_constants_from_survey():
    """SURVEY.md A.10: swf/cwf/lambda for the two standard rates."""
    m = PortOracle(rate_in=192000, mode=2, size=90).tables()["misc"]
    assert abs(m[0] - 0.5824777) < 1e-7 and abs(m[1] - 0.81284666) < 1e-7 and abs(m[2] - 0.6592406) < 1e-7
    m = PortOracle(rate_in=240000, mode=2, size=90).tables()["misc"]
    assert abs(m[0] - 0.47715878) < 1e-7 and abs(m[1] - 0.8788171) < 1e-7
    assert m[3] == np.float32(0.4) * np.float32(32768.0)


def test_rate_out_differs_from_rate_in_under_post_downsample():
    """-o N: main does rate_in *= post_downsample (:1510) and leaves rate_out, so the filters are designed for
    rate_in while lp_real_f32's ticks run at rate_out/rate_out2 (:485).  The port follows the reference there
    (the reference's PCM of the golden case stereo384_o2_fm, and the live reference where it is built), and the
    result is NOT what rate_out = rate_in would give."""
    kw = CONFIGS["stereo384_o2"]
    cid, cfg, kind, stream, blocks = CASE_BY_ID["stereo384_o2_fm"]
    iq = make_input(cfg, kind, stream, blocks)
    a = GOLD[cid]
    assert np.array_equal(a, PortOracle(**kw).run(iq))
    if ref_available():
        live = make_input("stereo384_o2", "fm_stereo", 1, 2)
        assert np.array_equal(RefOracle(**kw).run(live), PortOracle(**kw).run(live))
    same_rate = dict(kw, rate_out=0)
    assert PortOracle(**same_rate).run(iq).size != a.size     # 8 ticks per 64 samples instead of 16


def test_block_split_invariance_when_no_quirk():
    """At 192 kHz the in-place quirk never fires, so the block size must not matter."""
    iq = make_input("stereo192", "random", 11, 2)
    whole = PortOracle(**CONFIGS["stereo192"]).run(iq, block_bytes=B)
    halves = PortOracle(**CONFIGS["stereo192"]).run(iq, block_bytes=B // 8)
    assert np.array_equal(whole, halves)


def test_quirk_matters_at_240k():
    """Sanity of the A.7 emulation switch: with it off the 240 kHz stereo PCM differs."""
    iq = make_input("stereo240", "random", 5, 3)
    kw = CONFIGS["stereo240"]
    a = PortOracle(inplace_quirk=1, **kw).run(iq)
    b = PortOracle(inplace_quirk=0, **kw).run(iq)
    assert a.shape == b.shape and not np.array_equal(a, b)
    assert np.array_equal(a[:6552], b[:6552])      # block 0 has no tick on its first sample


def test_closed_form_of_the_resampler_ticks_equals_the_reference_accumulator():
    """The generic tick path of the demod kernel places output frame f0+m of a sub-tile that starts at
    sample j0 on sample i = ((m+1)*fast - rem0 - 1) // slow, with phase0 + j0*slow = f0*fast + rem0
    (rtl_fm_player_b200/csrc/fmb_kernels.cu).  The reference walks (prev_lpr_index += slow) >= fast
    (src/rtl_fm_player.c:570-572).  Same ticks, same frame numbers, for any ratio and phase."""
    rng = np.random.default_rng(7)
    cases = [(48000, 240000, 0), (48000, 192000, 0), (44100, 250000, 0), (48000, 100000, 0), (1, 1, 0)]
    for _ in range(40):
        fast = int(rng.integers(2, 400000))
        slow = int(rng.integers(1, fast))
        cases.append((slow, fast, int(rng.integers(0, fast))))
    for slow, fast, phase0 in cases:
        n, sub = 16384, 2048
        want, p, frame = {}, phase0, 0                      # the reference loop over one block
        for i in range(n):
            p += slow
            if p >= fast:
                p -= fast
                want[frame] = i
                frame += 1
        got = {}
        for j0 in range(0, n, sub):                         # the kernel's per-sub-tile closed form
            a0 = phase0 + j0 * slow
            f0, rem0 = divmod(a0, fast)
            m = 0
            while True:
                i = ((m + 1) * fast - rem0 - 1) // slow
                if i >= sub:
                    break
                assert f0 + m not in got
                got[f0 + m] = j0 + i
                m += 1
        assert got == want, (slow, fast, phase0)
