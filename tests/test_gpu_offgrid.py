"""The CUDA path off the golden grid: every block-start resampler phase a handle visits or may import, every block
size, the rate limits fmb_create checks, and the output stage.  The golden cases (tests/vectors.py) start at phase 0
and run 2-7 blocks of 262 144 bytes; the accepted configuration space is much larger, and so is the set of kernel
paths it reaches (the generic tick path at imported phases, dec_c0 != 0 on a 4:1 ratio, the in-place quirk at any
phase, sub-tile counts other than 8, blocks with no output at all, the de-emphasis repair loop on programme material).

Bar, as in test_gpu_parity.py: int16 PCM bit for bit against the C restatement (oracle/fm_oracle.c, PortOracle);
the discriminator and decoder outputs (fmb_debug_read) bit for bit on the few-stream runs.  Where the reference
build (oracle/_ref) exists, every configuration introduced here is also pinned oracle-against-reference once,
from phase 0, because the restatement is pinned to the reference only on the golden configurations.

Each sweep prints how many points it ran and how many it refused, and why (pytest -s)."""
import ctypes as C
import math
import random

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from oracle.oracle_py import REF_BLOCK, PortOracle, RefOracle, ref_available
from rtl_fm_player_b200 import _lib as L
from vectors import CONFIGS

pytestmark = pytest.mark.gpu

B = 262144
NSUB = 2048                                       # demodulated samples per sub-tile (FMB_NSUB)
QUANTUM = 32768                                   # FMB_BLOCK_QUANTUM: one sub-tile of IQ bytes
# fmb_create evaluates a sub-tile's tick schedule in 32-bit arithmetic and refuses (FMB_NSUB + FMB_NT + 2) * fast >= 2^32
LIMIT_FAST = ((1 << 32) - 1) // (NSUB + 256 + 2)

OFFGRID = dict(CONFIGS)
OFFGRID.update({
    "stereo250_44": dict(rate_in=250000, rate_out2=44100, mode=2, size=90, offset_tuning=0),
    "stereo_limit": dict(rate_in=LIMIT_FAST, rate_out2=48000, mode=2, size=90, offset_tuning=0),
    "mono_limit": dict(rate_in=LIMIT_FAST, rate_out2=48000, mode=1, size=128, offset_tuning=1),
    "mono_limit_every": dict(rate_in=LIMIT_FAST, rate_out2=LIMIT_FAST, mode=1, size=128, offset_tuning=0),
    "mono192_every": dict(rate_in=192000, rate_out2=192000, mode=1, size=90, offset_tuning=0),
    "stereo200_100": dict(rate_in=200000, rate_out2=100000, mode=2, size=90, offset_tuning=1),
    "mono192_50": dict(rate_in=192000, rate_out2=50, mode=1, size=128, offset_tuning=0),
    "stereo192_93": dict(rate_in=192000, rate_out2=93, mode=2, size=90, offset_tuning=0),
    "stereo192_5ms": dict(rate_in=192000, rate_out2=48000, mode=2, size=90, offset_tuning=0, deemph=0.005),
    "mono240_20ms": dict(rate_in=240000, rate_out2=48000, mode=1, size=128, offset_tuning=0, deemph=0.020),
})


def fast_of(kw):
    return kw.get("rate_out") or kw["rate_in"]


def capture(kw, kind, stream, n_bytes):
    return R.synth.capture(kind, stream, kw["rate_in"], kw.get("offset_tuning", 0), n_bytes // 2)


def make_cfg(kw, **extra):
    c = dict(kw)
    c.update(extra)
    return R.DemodConfig(**c)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def ref_pin(kw, iq, bb):
    """The restatement against the reference's own code, block by block from phase 0 (where that build exists and
    the block fits the reference's buffer)."""
    if not ref_available() or bb > REF_BLOCK:
        return
    ref, port = RefOracle(**kw), PortOracle(**kw)
    for b in range(iq.size // bb):
        blk = iq[b * bb:(b + 1) * bb]
        assert np.array_equal(port.block(blk), ref.block(blk)), f"oracle differs from the reference build, block {b}"


def refused(code, fn, *a):
    with pytest.raises(R.FmbError) as e:
        fn(*a)
    assert e.value.code == code, str(e.value)


# ---- the resampler schedule and the reference's in-place index walk, restated -----------------------------------

def step_of(kw, bb):
    return (bb // 16) * kw["rate_out2"] % fast_of(kw)


def cycle(kw, phase0=0, bb=B):
    """Block-start phases (prev_lpr_index) a handle visits from phase0, in order: phase += n_dem*slow mod fast."""
    fast = fast_of(kw)
    n = fast // math.gcd(step_of(kw, bb), fast)
    return ((phase0 + np.arange(n, dtype=np.int64) * step_of(kw, bb)) % fast).tolist()


def walk_hazard(fast, slow, n_dem, phases):
    """For each block-start phase: does the reference's stereo decoder (:570-597), which writes its outputs ib[o],
    ib[o+1] into the buffer it reads ib[i] from, overwrite an input it has not read yet -- other than the case the
    kernels emulate, a tick on sample 0 that overwrites sample 1?  The walk itself, sample by sample: prev_lpr_index
    += slow; a tick when it reaches fast (at most one per sample, slow <= fast), output index o = 2 x earlier ticks."""
    phases = np.asarray(phases, dtype=np.int64)
    out = np.zeros(len(phases), dtype=bool)
    i = np.arange(n_dem, dtype=np.int64)
    rows = max(1, (1 << 21) // n_dem)
    for a in range(0, len(phases), rows):
        ticks = (phases[a:a + rows, None] + slow * (i + 1)) // fast       # ticks up to and including sample i
        tick = np.diff(ticks, axis=1, prepend=0) > 0                      # phase < fast: no tick before sample 0
        o = 2 * (ticks - 1)
        out[a:a + rows] = (tick & (o + 1 > i) & (i > 0)).any(axis=1)
    return out


def cycle_refused(kw, phase0, bb):
    """fmb_create (phase 0) / fmb_set_state (imported phase) must refuse exactly when the cycle holds a hazard."""
    if kw["mode"] != 2 or kw["rate_out2"] <= 0:
        return False
    return bool(walk_hazard(fast_of(kw), kw["rate_out2"], bb // 16, cycle(kw, phase0, bb)).any())


# ---- state hand-over ----------------------------------------------------------------------------------------------

_FLOAT_BYTES = L.FmbStreamState.raw_valid.offset     # fmb_stream_state and the oracle's state agree up to deemph_r


def from_oracle(st):
    """The oracle's float state as an fmb_stream_state without raw bytes: the kernels rebuild the channel filter's
    history from the floats (chan_fir_from_state), as for a state taken from a reference demod_state."""
    f = L.FmbStreamState()
    C.memmove(C.addressof(f), C.addressof(st), _FLOAT_BYTES)
    f.raw_valid = 0
    return f


def assert_state_equal(g, o, mode, where):
    names = ["lowpass_tb", "pre_r", "pre_j", "br", "deemph_l"] + (["bm", "bs", "pp", "deemph_r"] if mode == 2 else [])
    for f in names:
        gf = np.array(getattr(g, f), dtype=np.float32, ndmin=1)
        of = np.array(getattr(o, "tb" if f == "lowpass_tb" else f), dtype=np.float32, ndmin=1)
        assert np.array_equal(bits(gf), bits(of)), f"{where}: carried {f} differs from the oracle's"


# ---- 1. phase sweep -------------------------------------------------------------------------------------------------

SWEEP = ["stereo240", "stereo170_44", "stereo250_44", "stereo96_48", "mono240_32", "mono240", "stereo384_o2",
         "stereo480_o2", "mono384_o2", "stereo192", "mono192"]


def sweep_phases(kw, limit=500, sample=100, edges=40, seed=1):
    """The block-start cycle from phase 0 when it has at most `limit` phases, else its boundary phases plus a seeded
    sample; always the imported phases around the tick grid: the multiples of slow (dec_c0 = 1, 2, .. when the ratio
    is integral) and 1, slow-1, fast-slow (the first with a tick on sample 0), fast-slow+-1 and fast-1."""
    fast, slow = fast_of(kw), kw["rate_out2"]
    cyc = cycle(kw)
    extra = [k * slow for k in range(1, fast // slow + 1) if k * slow < fast]
    extra += [1, slow - 1, fast - slow - 1, fast - slow, fast - slow + 1, fast - 1]
    if len(cyc) <= limit:
        base = cyc
    else:
        edge = [p for p in cyc if p < slow or p >= fast - slow - 400]
        base = sorted(set(cyc[:8] + edge[:edges] + edge[-edges:] + random.Random(seed).sample(cyc, sample)))
    seen, out = set(), []
    for p in base + extra:
        if 0 <= p < fast and p not in seen:
            seen.add(p)
            out.append(p)
    return out


def run_phase_sweep(kw, phases, n, uniq, kind, ws_generic=True, bb=B, fma=False):
    """At every phase: the oracle and the handle are put into the same carried state and phase (fmo_set_state,
    fmb_set_state) and run one or two blocks; PCM, out counts, the next phase and, for few streams, the discriminator
    and decoder outputs must match.  The handle resumes twice from the same point: from a state built from the
    oracle's floats (raw_valid 0: chan_fir_from_state) and from the state it exported itself (raw_valid 1: raw tail).
    fma: the handle runs FMB_PRECISION_FMA and the oracle is the fused restatement.  Returns (ran, refused)."""
    mode, fast = kw["mode"], fast_of(kw)
    per = 2 if len(phases) <= 64 else 1
    nb = 3
    iq_u = np.stack([capture(kw, kind, s, (nb + per) * bb) for s in range(uniq)])
    rows = np.arange(n) % uniq
    blocks = [np.ascontiguousarray(iq_u[rows, b * bb:(b + 1) * bb]) for b in range(nb + per)]
    orc = [PortOracle(**kw, fma=fma) for _ in range(uniq)]
    debug = n <= 4
    ran = refused_n = 0
    precision = R.FMB_PRECISION_FMA if fma else R.FMB_PRECISION_EXACT
    with R.FmBatch(make_cfg(kw, n_streams=n, block_bytes=bb, precision=precision)) as fb:
        if debug:
            fb.debug_enable(True)
        pcm = fb.process(blocks[0])                              # non-trivial history in every stage
        for s in range(uniq):
            assert np.array_equal(pcm[s], orc[s].block(blocks[0][s]))
        for j, p in enumerate(phases):
            gst, _, done = fb.get_state()
            assert all(gst[s].raw_valid == 1 for s in range(n))
            ost = [o.state()[0] for o in orc]
            for s in range(uniq):
                assert_state_equal(gst[s], ost[s], mode, f"before phase {p}")
            if cycle_refused(kw, p, bb):
                with pytest.raises(R.FmbError) as e:
                    fb.set_state(gst, p, done)
                assert e.value.code == L.FMB_ERR_UNSUPPORTED, (p, str(e.value))
                refused_n += 1
                continue
            # the oracle's run from (state, p)
            want, stages = [], []
            for s, o in enumerate(orc):
                o.set_state(ost[s], p, done)
            for k in range(per):
                blk = blocks[1 + (j + k) % nb]
                res = [o.block(blk[s], stages=True) for s, o in enumerate(orc)]
                want.append([r[0] for r in res])
                stages.append([r[1] for r in res])
            want_next = orc[0].state()[1]
            assert want_next == (p + per * (bb // 16) * kw["rate_out2"]) % fast
            floats = (L.FmbStreamState * n)(*[from_oracle(ost[s % uniq]) for s in range(n)])
            for path, imp, raw in (("float state", floats, 0), ("exported state", gst, 1)):
                fb.set_state(imp, p, done)
                held, ph, _ = fb.get_state(0, 1)
                assert held[0].raw_valid == raw and ph == p, path
                cur = p
                for k in range(per):
                    blk = blocks[1 + (j + k) % nb]
                    if mode == 1:           # the warp-specialised kernel: 4:1 at phase 0, else its generic tick path
                        dec4 = cur == 0 and fast == 4 * kw["rate_out2"]
                        name = "fmb_mono_ws_kernel" if (ws_generic or dec4) else "fmb_demod_kernel"
                        assert fb.kernel_name() == name, (p, k)
                    cur = (cur + (bb // 16) * kw["rate_out2"]) % fast
                    assert fb.next_out_count() == len(want[k][0]), (path, p, k)
                    got = fb.process(blk)
                    for s in range(n):
                        assert np.array_equal(got[s], want[k][s % uniq]), f"{path}, phase {p}, block {k}, stream {s}"
                    if debug:
                        dem, lr = fb.debug_read()
                        for s in range(n):
                            st = stages[k][s % uniq]
                            assert np.array_equal(bits(dem[s]), bits(st["dem"])), f"{path}, phase {p}: discriminator"
                            assert np.array_equal(bits(lr[s, :len(st["lr"])]), bits(st["lr"])), f"{path}, phase {p}: decoder"
                st_after, ph, _ = fb.get_state(0, 1)
                assert ph == want_next and st_after[0].raw_valid == 1, path
            ran += 1
    return ran, refused_n


@pytest.mark.parametrize("regime", ["few", "batch"])
@pytest.mark.parametrize("name", SWEEP)
def test_every_block_start_phase_resumes_bit_exactly(monkeypatch, name, regime):
    """Few streams: the static split, every sub-tile but a stream's first entered through a recomputed lead-in.
    Batch: more (stream, sub-tile) units than resident CTAs, handed out through the ticket counter (whole streams,
    then 2-sub-tile runs); a seeded part of the long cycles."""
    kw = OFFGRID[name]
    kind = "fm_stereo" if kw["mode"] == 2 else "fm_mono"
    if regime == "few":
        phases = sweep_phases(kw)
        ran, ref_n = run_phase_sweep(kw, phases, 3, 3, kind)
    else:
        monkeypatch.setenv("FMB_CHUNK", "2")
        monkeypatch.setenv("FMB_TAIL_PCT", "50")
        phases = sweep_phases(kw, limit=24, sample=16, edges=8)
        ran, ref_n = run_phase_sweep(kw, phases, 128, 4, "random")
    print(f"\n{name} {regime}: {len(phases)} phases, {ran} bit-exact on both resume paths, {ref_n} refused "
          f"(in-place hazard on their cycle)")
    assert ran > 0


MONO = ["mono240_32", "mono240", "mono384_o2", "mono192"]


@pytest.mark.parametrize("name", MONO)
def test_mono_phase_sweep_without_the_warp_specialised_generic_path(monkeypatch, name):
    """FMB_WS_GENERIC=0: mono off the 4:1 fast path runs fmb_demod_kernel's generic tick path."""
    monkeypatch.setenv("FMB_WS_GENERIC", "0")
    kw = OFFGRID[name]
    phases = sweep_phases(kw)
    ran, ref_n = run_phase_sweep(kw, phases, 3, 3, "random", ws_generic=False)
    print(f"\n{name} FMB_WS_GENERIC=0: {len(phases)} phases, {ran} bit-exact, {ref_n} refused")
    assert ran == len(phases) and ref_n == 0


@pytest.mark.parametrize("name", ["stereo250_44"])
def test_new_sweep_configurations_oracle_equals_reference_build(name):
    if not ref_available():
        pytest.skip("the reference build (oracle/_ref) is not present")
    kw = OFFGRID[name]
    ref_pin(kw, capture(kw, "fm_stereo", 3, 4 * B), B)


# ---- 2. the in-place refusal is exact -----------------------------------------------------------------------------

def refusal_grid():
    """Stereo (rate_in, rate_out, rate_out2, block_bytes) with rate_out/rate_out2 in [2, 3.2]."""
    pts = []
    for slow in (32000, 44100, 48000):
        for r in np.linspace(2.0, 3.2, 13):
            for bb in (QUANTUM, 3 * QUANTUM, B):
                step = 1000 if bb == B else 100                     # keeps the full-size blocks' cycles short
                fast = int(round(slow * r / step)) * step
                if 2 * slow <= fast:
                    pts.append((fast, 0, slow, bb))
    pts += [(2 * f, f, s, bb) for f, s, bb in ((100000, 48000, B), (128000, 48000, B), (112000, 44100, QUANTUM),
                                                (140000, 48000, 3 * QUANTUM))]    # -o 2: ticks at rate_out
    return pts


def test_inplace_refusal_is_exactly_the_walks_verdict():
    """fmb_create refuses a stereo configuration exactly when its block-start cycle from phase 0 holds an in-place
    hazard by the walk; fmb_set_state refuses an imported phase exactly when the cycle from that phase holds one.
    Then, per (rate_out2, block_bytes), the accepted configuration with the lowest ratio runs bit-exactly over (at
    most 6 blocks of) its cycle from phase 0 and from its highest accepted imported phase."""
    n_cfg = n_cfg_ref = n_imp = n_imp_ref = 0
    lowest = {}                                    # (rate_out2, block_bytes, -o) -> (ratio, kw, highest accepted import)
    for rate_in, rate_out, slow, bb in refusal_grid():
        kw = dict(rate_in=rate_in, rate_out=rate_out, rate_out2=slow, mode=2, size=90, offset_tuning=0)
        fast = fast_of(kw)
        n_cfg += 1
        if cycle_refused(kw, 0, bb):
            n_cfg_ref += 1
            refused(L.FMB_ERR_UNSUPPORTED, R.FmBatch, make_cfg(kw, block_bytes=bb))
            continue
        top = 0
        with R.FmBatch(make_cfg(kw, block_bytes=bb)) as fb:
            st, _, _ = fb.get_state()
            edge = 2 * fast - 3 * slow                 # about here tick 1 of a block moves onto sample 2
            for p in sorted({1, slow - 1, fast // 2, fast - slow, fast - 1, edge - 1, edge, edge + 1}):
                if not 0 < p < fast:
                    continue
                n_imp += 1
                if cycle_refused(kw, p, bb):
                    n_imp_ref += 1
                    refused(L.FMB_ERR_UNSUPPORTED, fb.set_state, st, p, 0)
                else:
                    fb.set_state(st, p, 0)
                    assert fb.get_state(0, 1)[1] == p
                    top = max(top, p)
        key = (slow, bb, rate_out > 0)
        if key not in lowest or fast < fast_of(lowest[key][1]):
            lowest[key] = (fast / slow, kw, top)
    print(f"\nrefusal grid: {n_cfg} configurations, {n_cfg_ref} refused by fmb_create; {n_imp} imported phases on the "
          f"accepted ones, {n_imp_ref} refused by fmb_set_state (cycle holds an in-place hazard)")
    assert 0 < n_cfg_ref < n_cfg and 0 < n_imp_ref < n_imp
    ran = 0
    for (slow, bb, _), (ratio, kw, top) in sorted(lowest.items()):
        iq = np.stack([capture(kw, "random", s, 7 * bb) for s in range(2)])
        ref_pin(kw, iq[0], bb)
        for p in sorted({0, top}):
            nblk = min(len(cycle(kw, p, bb)), 6)
            want = []
            for s in range(2):
                o = PortOracle(**kw)
                o.block(iq[s, :bb])
                o.set_state(o.state()[0], p, 1)
                want.append(np.concatenate([o.block(iq[s, b * bb:(b + 1) * bb]) for b in range(1, nblk + 1)]))
            with R.FmBatch(make_cfg(kw, n_streams=2, block_bytes=bb)) as fb:
                fb.process(np.ascontiguousarray(iq[:, :bb]))
                st, _, _ = fb.get_state()
                fb.set_state(st, p, 1)
                got = np.concatenate([fb.process(np.ascontiguousarray(iq[:, b * bb:(b + 1) * bb]))
                                      for b in range(1, nblk + 1)], axis=1)
            for s in range(2):
                assert np.array_equal(got[s], want[s]), (kw, bb, p, s)
            ran += 1
    print(f"lowest accepted ratios run bit-exactly: {ran} (configuration, phase) points")


# ---- 3. block sizes -----------------------------------------------------------------------------------------------

BLOCK_K = [1, 2, 3, 5, 7, 8, 9, 16]
BLOCK_CFGS = ["stereo192", "stereo192_128", "stereo240", "stereo170_44", "mono192", "mono240_32"]


def run_block_size_sweep(monkeypatch, kw, k, fma=False):
    """block_bytes = 32768*k: k sub-tiles per stream and block.  Several carried blocks against
    PortOracle.run(block_bytes=...), for every `segments` that divides k (and the automatic choice) on a few streams,
    and for a batch with more units than resident CTAs handed out through the ticket counter in 1-sub-tile runs.
    fma: FMB_PRECISION_FMA against the fused restatement.  Returns (segments values, batch streams)."""
    bb = QUANTUM * k
    nblk = 6
    kind = "fm_stereo" if kw["mode"] == 2 else "fm_mono"
    precision = R.FMB_PRECISION_FMA if fma else R.FMB_PRECISION_EXACT
    iq = np.stack([capture(kw, kind if s % 2 == 0 else "random", s, nblk * bb) for s in range(4)])
    want = [PortOracle(**kw, fma=fma).run(iq[s], block_bytes=bb) for s in range(4)]
    ref_pin(kw, iq[0], bb)
    segs = sorted(set([0] + [s for s in (1, 2, 4, 8, k) if k % s == 0]))
    for seg in segs:
        with R.FmBatch(make_cfg(kw, n_streams=3, block_bytes=bb, segments=seg, precision=precision)) as fb:
            if kw["mode"] == 1:             # a forced segmentation has no warp-specialised plan
                assert fb.kernel_name() == ("fmb_mono_ws_kernel" if seg == 0 else "fmb_demod_kernel")
            pcm = fb.run(iq[:3])
        for s in range(3):
            assert np.array_equal(pcm[s], want[s]), (k, seg, s)
    monkeypatch.setenv("FMB_CHUNK", "1")
    monkeypatch.setenv("FMB_TAIL_PCT", "50")
    n = -(-1024 // k)
    rows = np.arange(n) % 4
    with R.FmBatch(make_cfg(kw, n_streams=n, block_bytes=bb, precision=precision)) as fb:
        got = [fb.process(np.ascontiguousarray(iq[rows, b * bb:(b + 1) * bb])) for b in range(4)]
    got = np.concatenate(got, axis=1)
    for s in range(n):
        assert np.array_equal(got[s], want[s % 4][:got.shape[1]]), (k, "batch", s)
    return segs, n


@pytest.mark.parametrize("k", BLOCK_K)
@pytest.mark.parametrize("name", BLOCK_CFGS)
def test_block_size_sweep(monkeypatch, name, k):
    run_block_size_sweep(monkeypatch, OFFGRID[name], k)


# ---- 4. rate boundaries -------------------------------------------------------------------------------------------

def run_exact(kw, kind, nblk, n=2, bb=B, **extra):
    """n streams x nblk carried blocks against the oracle, out counts included; returns the PCM of stream 0."""
    iq = np.stack([capture(kw, kind, s, nblk * bb) for s in range(n)])
    orc = [PortOracle(**kw) for _ in range(n)]
    out = []
    with R.FmBatch(make_cfg(kw, n_streams=n, block_bytes=bb, **extra)) as fb:
        fb.debug_enable(True)
        for b in range(nblk):
            blk = np.ascontiguousarray(iq[:, b * bb:(b + 1) * bb])
            res = [o.block(blk[s], stages=True) for s, o in enumerate(orc)]
            assert fb.next_out_count() == len(res[0][0]), f"block {b}: out count"
            pcm = fb.process(blk)
            dem, lr = fb.debug_read()
            for s in range(n):
                assert np.array_equal(pcm[s], res[s][0]), f"block {b}, stream {s}: PCM"
                assert np.array_equal(bits(dem[s]), bits(res[s][1]["dem"])), f"block {b}, stream {s}: discriminator"
                assert np.array_equal(bits(lr[s, :len(res[s][1]["lr"])]), bits(res[s][1]["lr"])), f"block {b}: decoder"
            out.append(pcm[0])
    ref_pin(kw, iq[0], bb)
    return np.concatenate(out)


@pytest.mark.parametrize("name", ["stereo_limit", "mono_limit", "mono_limit_every"])
def test_highest_rate_fmb_create_accepts(name):
    """The largest fast rate the 32-bit tick schedule allows is accepted and exact (mono with every sample a tick
    too: 2048 ticks per sub-tile, the warp-specialised kernel's 128-thread back role in 16 rounds); one more is
    refused."""
    kw = OFFGRID[name]
    run_exact(kw, "random" if kw["mode"] == 1 else "fm_stereo", 3)
    over = dict(kw, rate_in=LIMIT_FAST + 1, rate_out2=min(kw["rate_out2"], LIMIT_FAST + 1))
    refused(L.FMB_ERR_UNSUPPORTED, R.FmBatch, make_cfg(over))
    o2 = dict(kw, rate_in=2 * (LIMIT_FAST + 1), rate_out=LIMIT_FAST + 1)            # the same limit on rate_out (-o 2)
    refused(L.FMB_ERR_UNSUPPORTED, R.FmBatch, make_cfg(o2))


@pytest.mark.parametrize("name", ["mono192_every", "mono_limit_every"])
@pytest.mark.parametrize("ws", ["1", "0"])
def test_mono_every_sample_a_tick(monkeypatch, name, ws):
    monkeypatch.setenv("FMB_WS", ws)
    kw = OFFGRID[name]
    with R.FmBatch(make_cfg(kw)) as fb:
        assert fb.kernel_name() == ("fmb_mono_ws_kernel" if ws == "1" else "fmb_demod_kernel")
        assert fb.next_out_count() == B // 16
    run_exact(kw, "fm_mono", 3)


def test_stereo_ratio_two_is_accepted_and_one_below_is_refused():
    for kw in (OFFGRID["stereo96_48"], OFFGRID["stereo200_100"]):
        run_exact(kw, "random", 3)
        run_exact(kw, "fm_stereo", 3, bb=QUANTUM)
        below = dict(kw, rate_in=2 * kw["rate_out2"] - 1)
        refused(L.FMB_ERR_UNSUPPORTED, R.FmBatch, make_cfg(below))
        below_o2 = dict(kw, rate_in=2 * kw["rate_in"], rate_out=2 * kw["rate_out2"] - 1)
        refused(L.FMB_ERR_UNSUPPORTED, R.FmBatch, make_cfg(below_o2))


@pytest.mark.parametrize("name", ["mono192_50", "stereo192_93"])
def test_blocks_with_zero_or_one_output(name):
    """rate_out2 so low that a 32768-byte block (2048 demodulated samples) holds 0 or 1 ticks: the out count of every
    block is the oracle's, empty blocks included, and the PCM matches."""
    kw = OFFGRID[name]
    nblk = 10
    counts = []
    iq = np.stack([capture(kw, "random", s, nblk * QUANTUM) for s in range(2)])
    orc = [PortOracle(**kw) for _ in range(2)]
    with R.FmBatch(make_cfg(kw, n_streams=2, block_bytes=QUANTUM)) as fb:
        for b in range(nblk):
            blk = np.ascontiguousarray(iq[:, b * QUANTUM:(b + 1) * QUANTUM])
            want = [o.block(blk[s]) for s, o in enumerate(orc)]
            counts.append(fb.next_out_count())
            assert counts[-1] == len(want[0]), b
            pcm = fb.process(blk)
            for s in range(2):
                assert np.array_equal(pcm[s], want[s]), (b, s)
    per_tick = 2 if kw["mode"] == 2 else 1
    assert set(counts) == {0, per_tick}, counts
    ref_pin(kw, iq[0], QUANTUM)


# ---- 5. output stage ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("volume", [0.0, -0.4, -1.5, 40.0])
@pytest.mark.parametrize("name,kind", [("stereo192", "fm_stereo"), ("stereo240", "random"), ("mono240", "fm_mono")])
def test_volume_edges(name, kind, volume):
    """Volume 0 (all zeros), negative (the clamp is asymmetric: -32768 / 32767) and 40 (nearly every value clamps)."""
    kw = dict(OFFGRID[name], volume=volume)
    pcm = run_exact(kw, kind, 3)
    if volume == 0.0:
        assert not pcm.any()
    if volume == 40.0:                             # both ends of the clamp reached
        assert (pcm == 32767).any() and (pcm == -32768).any()


VOLS = [0.4, -1.5, 40.0, 0.0, 0.7, -0.4]


def oracle_with_volume_changes(kw, iq, vols):
    """One oracle per block, each taking over its predecessor's carried state (PortOracle fixes the volume)."""
    out, prev = [], None
    for b, v in enumerate(vols):
        o = PortOracle(**dict(kw, volume=v))
        if prev is not None:
            o.set_state(*prev.state())
        out.append(o.block(iq[b * B:(b + 1) * B]))
        prev = o
    return out


def test_set_volume_between_steps_and_between_pipelined_submits():
    """fmb_set_volume takes effect from the next process call (fmb.h).  On the pipelined path that is the next
    fmb_submit: the steps already submitted -- up to FMB_PIPE_DEPTH in flight -- keep the volume they were submitted
    with, so a volume change lands on a block boundary in submission order."""
    import torch
    kw = OFFGRID["stereo240"]
    n = 3
    iq = np.stack([capture(kw, "fm_stereo", s, len(VOLS) * B) for s in range(n)])
    want = [oracle_with_volume_changes(kw, iq[s], VOLS) for s in range(n)]
    with R.FmBatch(make_cfg(kw, n_streams=n, volume=VOLS[0])) as fb:
        for b, v in enumerate(VOLS):
            fb.set_volume(v)
            pcm = fb.process(np.ascontiguousarray(iq[:, b * B:(b + 1) * B]))
            for s in range(n):
                assert np.array_equal(pcm[s], want[s][b]), ("process", b, s)
    with R.FmBatch(make_cfg(kw, n_streams=n, volume=VOLS[0])) as fb:
        pitch = (fb.max_out + 7) & ~7
        hin = [torch.from_numpy(iq[:, b * B:(b + 1) * B].copy()).pin_memory() for b in range(len(VOLS))]
        hout = [torch.zeros((n, pitch), dtype=torch.int16).pin_memory() for _ in VOLS]
        counts, tickets = [], []
        for b, v in enumerate(VOLS):
            if len(tickets) == L.FMB_PIPE_DEPTH:
                fb.wait(tickets.pop(0))
            fb.set_volume(v)                       # with FMB_PIPE_DEPTH steps still in flight from b >= 3
            counts.append(fb.next_out_count())
            tickets.append(fb.submit(hin[b].data_ptr(), B, hout[b].data_ptr(), pitch))
        for t in tickets:
            fb.wait(t)
    for b in range(len(VOLS)):
        for s in range(n):
            assert np.array_equal(hout[b].numpy()[s, :counts[b]], want[s][b]), ("submit", b, s)


def test_explicit_deemph_lambda_is_used():
    """deemph_lambda > 0 replaces the pole computed from deemph (what the drop-in passes).  The handle is given the
    pole of a 5 ms constant beside a 50 us `deemph`; the oracle computes the 5 ms pole itself."""
    kw5 = OFFGRID["stereo192_5ms"]
    lam = float(PortOracle(**kw5).tables()["misc"][2])
    iq = np.stack([capture(kw5, "fm_stereo", s, 3 * B) for s in range(2)])
    with R.FmBatch(make_cfg(kw5, n_streams=2, deemph=0.000050, deemph_lambda=lam)) as fb:
        assert fb.tables()["misc"][2] == np.float32(lam)
        pcm = fb.run(iq)
    for s in range(2):
        assert np.array_equal(pcm[s], PortOracle(**kw5).run(iq[s])), s
    kw = OFFGRID["stereo192"]                      # the pole the drop-in passes for the default constant
    lam50 = float(PortOracle(**kw).tables()["misc"][2])
    with R.FmBatch(make_cfg(kw, n_streams=2, deemph_lambda=lam50)) as fb:
        pcm = fb.run(iq)
    for s in range(2):
        assert np.array_equal(pcm[s], PortOracle(**kw).run(iq[s])), s


@pytest.mark.parametrize("name,kind", [("stereo192_5ms", "fm_stereo"), ("mono240_20ms", "fm_mono")])
def test_deemphasis_pole_close_to_one_runs_the_repair_loop_and_stays_exact(name, kind):
    """A pole close to 1 keeps the speculative IIR from merging within its warm-up on programme material: the
    sequential repair runs on ordinary blocks (not only on digital silence), and the PCM is still the oracle's."""
    kw = OFFGRID[name]
    n, nblk = 4, 4
    iq = np.stack([capture(kw, kind, s, nblk * B) for s in range(n)])
    with R.FmBatch(make_cfg(kw, n_streams=n)) as fb:
        pcm = fb.process(np.ascontiguousarray(iq[:, :B]))
        first = fb.deemph_fallbacks()
        rest = [fb.process(np.ascontiguousarray(iq[:, b * B:(b + 1) * B])) for b in range(1, nblk)]
        total = fb.deemph_fallbacks()
    pcm = np.concatenate([pcm] + rest, axis=1)
    for s in range(n):
        assert np.array_equal(pcm[s], PortOracle(**kw).run(iq[s])), s
    print(f"\n{name}: {total} de-emphasis chunks repaired sequentially ({first} in the first block)")
    assert total > first, (first, total)
    ref_pin(kw, iq[0], B)
