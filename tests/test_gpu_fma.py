"""FMB_PRECISION_FMA bit for bit.  The FMA kernels fuse exactly the FIR multiply-adds (channel FIR taps 1-15, the
decoder's vm/vp/vs, the symmetric FIRs of the second low-pass and of mono), in the reference's order; everything else
is rounded as in exact mode.  The fused restatement (oracle/fm_oracle.c built with FMO_FMA, PortOracle(fma=True))
computes the same thing on the CPU, and tests/test_oracle_fma.py pins it within +-1 LSB of the reference.  So every
comparison here is exact: int16 PCM, the discriminator and decoder taps (fmb_debug_read) on few-stream runs, and the
carried state (fmb_get_state), against the fused restatement.

  * every one of the 18 FMA kernel instantiations, named in INSTANTIATIONS, on programme material and random bytes;
  * every golden case's input and the three 10 s captures;
  * work assignment: segments, the ticketed split, overlapping and plain back-to-back launches, stream counts;
  * off the golden grid: block-start phase sweeps (both resume paths), block sizes 32768*k;
  * the multi-GPU host.

Under pytest -s each test prints what it ran."""
import json
import os

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from oracle.oracle_py import PortOracle
from test_gpu_multi import _devices
from test_gpu_parity import run_back_to_back
from test_gpu_offgrid import (OFFGRID, QUANTUM, assert_state_equal, bits, capture, fast_of, run_block_size_sweep,
                              run_phase_sweep, sweep_phases)
from vectors import B, CASES, CONFIGS, LONG_CASES, long_capture_bytes, make_input, sha

GPU = pytest.mark.gpu
FMA = R.FMB_PRECISION_FMA
HERE = os.path.dirname(os.path.abspath(__file__))
META = json.load(open(os.path.join(HERE, "golden", "golden_meta.json")))

# offset-tuning (ROT=false) and size variants that tests/vectors.py does not define
FMA_CONFIGS = dict(OFFGRID)
FMA_CONFIGS.update({
    "stereo192_128_off": dict(rate_in=192000, rate_out2=48000, mode=2, size=128, offset_tuning=1),
    "mono192_90_off": dict(rate_in=192000, rate_out2=48000, mode=1, size=90, offset_tuning=1),
    "drop192_off": dict(rate_in=192000, rate_out2=48000, mode=0, size=90, offset_tuning=1),
    "mono240_90": dict(rate_in=240000, rate_out2=48000, mode=1, size=90, offset_tuning=0),
    "mono240_90_off": dict(rate_in=240000, rate_out2=48000, mode=1, size=90, offset_tuning=1),
})

# (instantiation, configurations that run it, environment).  fmb_demod_kernel<MODE, S, ROT, FMA>: mono only with
# FMB_WS=0 (or FMB_WS_GENERIC=0 off the 4:1 ratio), mode 0 for lpr.mode 0 and for rate_out2 = 0.
# fmb_mono_ws_kernel<S, ROT, FMA, LIN>: LIN = the generic tick path, off the 4:1 ratio.
INSTANTIATIONS = [
    ("fmb_demod_kernel<0,2,true,true>", ["drop192", "nolpr192"], {}),
    ("fmb_demod_kernel<0,2,false,true>", ["drop192_off"], {}),
    ("fmb_demod_kernel<1,90,true,true>", ["mono192_90", "mono240_90"], {"FMB_WS": "0"}),
    ("fmb_demod_kernel<1,90,false,true>", ["mono192_90_off", "mono240_90_off"], {"FMB_WS": "0"}),
    ("fmb_demod_kernel<1,128,true,true>", ["mono192", "mono240_32"], {"FMB_WS": "0"}),
    ("fmb_demod_kernel<1,128,false,true>", ["mono240_off"], {"FMB_WS_GENERIC": "0"}),
    ("fmb_demod_kernel<2,90,true,true>", ["stereo192", "stereo240", "stereo170_44"], {}),
    ("fmb_demod_kernel<2,90,false,true>", ["stereo192_off", "stereo256_48"], {}),
    ("fmb_demod_kernel<2,128,true,true>", ["stereo192_128"], {}),
    ("fmb_demod_kernel<2,128,false,true>", ["stereo192_128_off"], {}),
    ("fmb_mono_ws_kernel<90,true,true,false>", ["mono192_90"], {}),
    ("fmb_mono_ws_kernel<90,true,true,true>", ["mono240_90"], {}),
    ("fmb_mono_ws_kernel<90,false,true,false>", ["mono192_90_off"], {}),
    ("fmb_mono_ws_kernel<90,false,true,true>", ["mono240_90_off"], {}),
    ("fmb_mono_ws_kernel<128,true,true,false>", ["mono192"], {}),
    ("fmb_mono_ws_kernel<128,true,true,true>", ["mono240", "mono240_32"], {}),
    ("fmb_mono_ws_kernel<128,false,true,false>", ["mono384_o2"], {}),
    ("fmb_mono_ws_kernel<128,false,true,true>", ["mono240_off"], {}),
]


def instantiation(kw, env):
    """The kernel template fmb_create / fmb_process pick for a configuration at phase 0 in FMA mode (fmb_api.cu,
    dispatch_demod in fmb_kernels.cu), restated."""
    mode = kw["mode"] if kw["rate_out2"] > 0 else 0
    size = kw["size"] if mode else 2
    rot = "false" if kw.get("offset_tuning", 0) else "true"
    dec4 = kw["rate_out2"] > 0 and fast_of(kw) == 4 * kw["rate_out2"]
    if mode == 1 and env.get("FMB_WS") != "0" and (dec4 or env.get("FMB_WS_GENERIC") != "0"):
        return f"fmb_mono_ws_kernel<{size},{rot},true,{'false' if dec4 else 'true'}>"
    return f"fmb_demod_kernel<{mode},{size},{rot},true>"


def test_the_table_names_every_fma_instantiation_once():
    names = [row[0] for row in INSTANTIATIONS]
    want = {f"fmb_demod_kernel<0,2,{r},true>" for r in ("true", "false")}
    want |= {f"fmb_demod_kernel<{m},{s},{r},true>" for m in (1, 2) for s in (90, 128) for r in ("true", "false")}
    want |= {f"fmb_mono_ws_kernel<{s},{r},true,{lin}>" for s in (90, 128) for r in ("true", "false")
             for lin in ("false", "true")}
    assert len(want) == 18 and len(names) == 18 and set(names) == want
    for name, cfgs, env in INSTANTIATIONS:
        for c in cfgs:
            assert instantiation(FMA_CONFIGS[c], env) == name, (name, c)


def fcfg(kw, **extra):
    c = dict(kw, precision=FMA)
    c.update(extra)
    return R.DemodConfig(**c)


def fused(kw):
    return PortOracle(**kw, fma=True)


def programme(kw):
    return "fm_stereo" if kw["mode"] != 1 else "fm_mono"


def check_state(fb, orc, kw, where):
    """fmb_get_state against the fused restatement's carried state, phase and block count."""
    gst, ph, done = fb.get_state()
    for s in range(len(gst)):
        o = orc[s % len(orc)]
        ost, oph, obl = o.state()
        assert (ph, done) == (oph, obl), where
        if kw["rate_out2"] > 0:
            assert_state_equal(gst[s], ost, kw["mode"], f"{where}, stream {s}")
        else:       # no decoder stage (lp_real_f32 skipped): the reference carries only these
            for g, f in (("lowpass_tb", "tb"), ("pre_r", "pre_r"), ("pre_j", "pre_j"), ("deemph_l", "deemph_l"),
                         ("deemph_r", "deemph_r")):
                a, b = (np.array(getattr(x, n), dtype=np.float32, ndmin=1) for x, n in ((gst[s], g), (ost, f)))
                assert np.array_equal(bits(a), bits(b)), f"{where}, stream {s}: carried {g}"


def run_model(kw, iq, bb=B, expect_kernel=None):
    """n = iq.shape[0] distinct streams, block by block, each against its own fused restatement: out counts, PCM, the
    discriminator and decoder taps (few streams) and the carried state after every block.  Returns (PCM of every
    stream, whether the exact build differs from the fused one somewhere on this input: a kernel that ignored FMA
    would then fail)."""
    n, nblk = iq.shape[0], iq.shape[1] // bb
    orc = [fused(kw) for _ in range(n)]
    exact = [PortOracle(**kw) for _ in range(n)]
    debug = n <= 4
    sees_fma = False
    out = []
    with R.FmBatch(fcfg(kw, n_streams=n, block_bytes=bb)) as fb:
        if expect_kernel:
            assert fb.kernel_name() == expect_kernel
        fb.debug_enable(debug)
        for b in range(nblk):
            blk = np.ascontiguousarray(iq[:, b * bb:(b + 1) * bb])
            res = [o.block(blk[s], stages=True) for s, o in enumerate(orc)]
            for s, e in enumerate(exact):
                p, st = e.block(blk[s], stages=True)
                sees_fma |= not (np.array_equal(bits(st["dem"]), bits(res[s][1]["dem"])) and
                                 np.array_equal(bits(st["lr"]), bits(res[s][1]["lr"])) and np.array_equal(p, res[s][0]))
            assert fb.next_out_count() == len(res[0][0]), f"block {b}: out count"
            pcm = fb.process(blk)
            for s in range(n):
                assert np.array_equal(pcm[s], res[s][0]), f"block {b}, stream {s}: PCM"
            if debug:
                dem, lr = fb.debug_read()
                for s in range(n):
                    st = res[s][1]
                    assert np.array_equal(bits(dem[s]), bits(st["dem"])), f"block {b}, stream {s}: discriminator"
                    assert np.array_equal(bits(lr[s, :len(st["lr"])]), bits(st["lr"])), f"block {b}, stream {s}: decoder"
            check_state(fb, orc, kw, f"after block {b}")
            out.append(pcm)
    return np.concatenate(out, axis=1), sees_fma


# ---- 1. every FMA instantiation -------------------------------------------------------------------------------------

@GPU
@pytest.mark.parametrize("name,cfgs,env", INSTANTIATIONS, ids=[r[0] for r in INSTANTIATIONS])
def test_every_fma_instantiation_equals_the_fused_restatement(monkeypatch, name, cfgs, env):
    """Each configuration of the row: one stream of programme material, then four distinct streams (programme
    material and random bytes), three carried blocks."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    kernel = name.split("<")[0]
    for c in cfgs:
        kw = FMA_CONFIGS[c]
        iq = np.stack([capture(kw, programme(kw) if s % 2 == 0 else "random", s, 3 * B) for s in range(4)])
        _, fma1 = run_model(kw, iq[:1], expect_kernel=kernel)
        _, fma4 = run_model(kw, iq, expect_kernel=kernel)
        assert fma1 and fma4, f"{c}: the exact and the fused restatement agree on this input, it cannot tell them apart"
    print(f"\n{name}: bit-exact on {', '.join(cfgs)} (n = 1 and 4, 3 blocks each)")


# ---- 2. the golden inputs -------------------------------------------------------------------------------------------

@GPU
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_golden_case_inputs_in_fma_mode(case):
    cid, cfg, kind, stream, blocks = case
    kw = CONFIGS[cfg]
    iq = make_input(cfg, kind, stream, blocks)
    assert sha(iq) == META["cases"][cid]["input_sha256"]
    batch = np.stack([iq] + [make_input(cfg, kind, stream + 17 * k, blocks) for k in range(1, 4)])
    pcm, _ = run_model(kw, batch[:1])
    assert pcm.shape[1] == sum(META["cases"][cid]["counts"])
    run_model(kw, batch)


@GPU
@pytest.mark.parametrize("case", LONG_CASES, ids=[c[0] for c in LONG_CASES])
def test_ten_second_captures_in_fma_mode(case):
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    iq = np.concatenate([iq, np.zeros(long_capture_bytes(cfg) - blocks * B, np.uint8)])
    with R.FmBatch(fcfg(CONFIGS[cfg], n_streams=1)) as fb:
        pcm = fb.run(iq[None, :])
    want = fused(CONFIGS[cfg]).run(iq)
    assert pcm.shape[1] == META["long"][cid]["n_pcm"] and np.array_equal(pcm[0], want)


# ---- 3. work assignment ---------------------------------------------------------------------------------------------

@GPU
@pytest.mark.parametrize("segs", [1, 2, 4, 8])
@pytest.mark.parametrize("cfgname,kind", [("stereo192", "random"), ("mono192", "fm_mono"), ("stereo240", "random")])
def test_fma_time_segmentation_does_not_change_the_result(cfgname, kind, segs):
    kw = CONFIGS[cfgname]
    blocks = 6 if cfgname == "stereo240" else 2
    iq = np.stack([make_input(cfgname, kind, s, blocks) for s in range(2)])
    with R.FmBatch(fcfg(kw, n_streams=2, segments=segs)) as fb:
        pcm = fb.run(iq)
    for s in range(2):
        assert np.array_equal(pcm[s], fused(kw).run(iq[s])), s


@GPU
@pytest.mark.parametrize("cfgname,kind,chunk,tail", [("stereo192", "fm_stereo", 1, 100), ("stereo192", "random", 4, 50),
                                                     ("mono192", "fm_mono", 2, 100), ("mono192", "fm_mono", 8, 100),
                                                     ("stereo240", "fm_stereo", 2, 60), ("stereo192", "fm_stereo", 0, 0),
                                                     ("mono240", "random", 2, 50)])
def test_fma_dynamic_work_assignment_does_not_change_the_result(monkeypatch, cfgname, kind, chunk, tail):
    monkeypatch.setenv("FMB_CHUNK", str(chunk))
    monkeypatch.setenv("FMB_TAIL_PCT", str(tail))
    n, uniq, blocks = 64, 8, 3
    c = CONFIGS[cfgname]
    iq = R.synth.batch(kind, n, c["rate_in"], c.get("offset_tuning", 0), blocks * B // 2, unique=uniq)
    with R.FmBatch(fcfg(c, n_streams=n)) as fb:
        pcm = fb.run(iq)
    for s in range(uniq):
        assert np.array_equal(pcm[s], fused(c).run(iq[s])), s
    assert np.array_equal(pcm.reshape(n // uniq, uniq, -1), np.broadcast_to(pcm[:uniq], (n // uniq, uniq, pcm.shape[1])))


@GPU
@pytest.mark.parametrize("cfgname,kind", [("stereo192", "fm_stereo"), ("mono192", "fm_mono"), ("stereo240", "random"),
                                          ("mono240", "fm_mono")])
@pytest.mark.parametrize("pdl", ["1", "0"])
def test_fma_back_to_back_full_batches(monkeypatch, cfgname, kind, pdl):
    """1024 streams x 6 blocks enqueued back to back with no host synchronisation: overlapping launches (FMB_PDL=1) and
    plain stream order (0).  16 distinct channels against the fused restatement, every replica equal to its original."""
    run_back_to_back(monkeypatch, cfgname, kind, pdl, fma=True)


@GPU
@pytest.mark.parametrize("n", [1, 31, 97, 1024])
@pytest.mark.parametrize("cfgname,kind", [("stereo192", "random"), ("mono240", "fm_mono")])
def test_fma_stream_counts(cfgname, kind, n):
    """Ragged batches and the size the benchmark times (1024 streams: 16 distinct channels repeated)."""
    c = CONFIGS[cfgname]
    uniq, blocks = min(n, 16), 2
    iq = R.synth.batch(kind, n, c["rate_in"], c.get("offset_tuning", 0), blocks * B // 2, unique=uniq)
    with R.FmBatch(fcfg(c, n_streams=n)) as fb:
        pcm = fb.run(iq)
        orc = [fused(c) for _ in range(uniq)]
        for s in range(uniq):
            assert np.array_equal(pcm[s], orc[s].run(iq[s])), s
        check_state(fb, orc, c, f"{n} streams")
    rows = np.arange(n) % uniq
    assert np.array_equal(pcm, pcm[rows])


# ---- 4. off the golden grid -----------------------------------------------------------------------------------------

@GPU
@pytest.mark.parametrize("regime", ["few", "batch"])
@pytest.mark.parametrize("name", ["stereo240", "stereo170_44", "mono240_32", "mono192"])
def test_fma_every_block_start_phase_resumes_bit_exactly(monkeypatch, name, regime):
    """The phase sweep of test_gpu_offgrid.py in FMA mode.  stereo240: the in-place quirk, whose scalar recomputation
    on thread 0 must round exactly like the packed FIRs; mono192: 4:1 mono at imported phases on the multiples of
    rate_out2 (dec_c0 != 0: the warp-specialised kernel's generic tick path).  Both resume paths: from the oracle's
    floats (chan_fir_from_state) and from the handle's exported state."""
    kw = OFFGRID[name]
    if regime == "few":
        phases = sweep_phases(kw)
        ran, ref_n = run_phase_sweep(kw, phases, 3, 3, programme(kw), fma=True)
    else:
        monkeypatch.setenv("FMB_CHUNK", "2")
        monkeypatch.setenv("FMB_TAIL_PCT", "50")
        phases = sweep_phases(kw, limit=24, sample=16, edges=8)
        ran, ref_n = run_phase_sweep(kw, phases, 128, 4, "random", fma=True)
    if name == "mono192":
        slow = kw["rate_out2"]
        assert any(p % slow == 0 and p > 0 for p in phases)
    print(f"\n{name} {regime} FMA: {len(phases)} phases, {ran} bit-exact on both resume paths, {ref_n} refused")
    assert ran > 0


@GPU
@pytest.mark.parametrize("k", [1, 3, 9])
@pytest.mark.parametrize("name", ["stereo192", "stereo240", "stereo192_128", "mono192", "mono240_32"])
def test_fma_block_size_sweep(monkeypatch, name, k):
    """block_bytes = 32768*k on a few streams for every `segments` that divides k (and the automatic choice), and in
    a ticketed batch of 1-sub-tile runs."""
    segs, n = run_block_size_sweep(monkeypatch, OFFGRID[name], k, fma=True)
    print(f"\n{name} FMA, block {QUANTUM * k} B: segments {segs} and a {n}-stream ticketed batch bit-exact")


# ---- 5. multi-GPU ---------------------------------------------------------------------------------------------------

@GPU
@pytest.mark.parametrize("cfgname,kind", [("stereo192", "fm_stereo"), ("mono240", "random")])
def test_fma_every_shard_matches_the_fused_restatement(cfgname, kind):
    devs = _devices(2)
    per, blocks = 8, 3
    n = per * len(devs)
    kw = CONFIGS[cfgname]
    iq = np.stack([make_input(cfgname, kind, s, blocks) for s in range(n)])
    with R.FmMulti(fcfg(kw, n_streams=n), devs) as fm:
        pcm = fm.run(iq)
    for s in range(n):
        assert np.array_equal(pcm[s], fused(kw).run(iq[s])), f"stream {s} (shard {s // per}, device {devs[s // per]})"
    print(f"\n{cfgname} FMA over devices {devs}: {n} streams bit-exact")
