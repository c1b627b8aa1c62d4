"""Parity of the CUDA path (through the C ABI, libfmb.so) with the CPU oracle and with the PCM
the reference's own code produced (tests/golden).  Bar: BIT-EXACT int16 PCM and bit-exact float
stage outputs in FMB_PRECISION_EXACT; +-1 LSB int16 in FMB_PRECISION_FMA (tolerance stated in
BASELINE.json's north_star for the floating-point stages)."""
import json
import os

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from oracle.oracle_py import PortOracle
from rtl_fm_player_b200 import _lib as L
from vectors import B, CASES, CONFIGS, LONG_CASES, REFUSED, long_capture_bytes, make_input, sha

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "golden.npz"))
META = json.load(open(os.path.join(HERE, "golden", "golden_meta.json")))


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# Stage outputs are compared BIT for bit.  The only leniency is the sign of an exact zero, and only for the vectors
# named here (digital silence / constant input, where the reference's early-return guards at :611-618 and :474 and
# our branch-free forms may disagree on -0.0 vs +0.0 in a value that no later stage can observe; the PCM is
# compared exactly everywhere).
SIGNED_ZERO_CASES = set()


def same_floats(a, b, cid=None):
    if np.array_equal(bits(a), bits(b)):
        return True
    return cid in SIGNED_ZERO_CASES and np.array_equal(np.asarray(a), np.asarray(b))


def cfg_for(name, **kw):
    c = dict(CONFIGS[name])
    c.update(kw)
    return R.DemodConfig(**c)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_cuda_pcm_equals_reference_golden_and_oracle_stages(case):
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    assert sha(iq) == META["cases"][cid]["input_sha256"]
    port = PortOracle(**CONFIGS[cfg])
    got = []
    with R.FmBatch(cfg_for(cfg, n_streams=1)) as fb:
        fb.debug_enable(True)
        for b in range(blocks):
            blk = iq[None, b * B:(b + 1) * B]
            assert fb.next_out_count() == META["cases"][cid]["counts"][b]
            pcm = fb.process(blk)
            dem, lr = fb.debug_read()
            p_or, st = port.block(blk[0], stages=True)
            assert same_floats(dem[0], st["dem"], cid), f"block {b}: discriminator output differs"
            assert same_floats(lr[0, :len(st["lr"])], st["lr"], cid), f"block {b}: decoder output differs"
            assert np.array_equal(pcm[0], p_or), f"block {b}: PCM differs from the oracle"
            got.append(pcm[0])
    assert np.array_equal(np.concatenate(got), GOLD[cid]), "PCM differs from the reference's own output"


@pytest.mark.parametrize("case", LONG_CASES, ids=[c[0] for c in LONG_CASES])
def test_configs_0_and_1_ten_second_capture(case):
    """BASELINE.json configs[0] (mono) and [1] (stereo): 10 s single-channel capture, sha256 of the
    PCM must equal the reference's.  configs[0] also at the literal default rate (rate_in 240 000 =
    DEFAULT_SAMPLE_RATE h:30, rotate path): 38 400 000 bytes, 146 full blocks."""
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    m = META["long"][cid]
    with R.FmBatch(cfg_for(cfg, n_streams=1)) as fb:
        pcm = fb.run(np.concatenate([iq, np.zeros(long_capture_bytes(cfg) - blocks * B, np.uint8)])[None, :])
    assert pcm.shape[1] == m["n_pcm"] and sha(pcm[0]) == m["pcm_sha256"]


def test_config_2_sixty_four_streams_forty_blocks_each_vs_its_own_oracle():
    """BASELINE.json configs[2] at the depth SURVEY s8d asks for: 64 distinct stereo channels x 40 block-steps
    (16 MiB per step, 640 MiB in all), every channel's whole PCM against its own oracle run."""
    from concurrent.futures import ThreadPoolExecutor
    n, blocks = 64, 40
    kw = CONFIGS["stereo192"]
    iq = R.synth.batch("fm_stereo", n, 192000, 0, blocks * B // 2, threads=min(16, os.cpu_count() or 1))
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        pcm = fb.run(iq)
        assert fb.deemph_fallbacks() < n * blocks       # the speculative IIR verified nearly everywhere
    assert pcm.shape == (n, blocks * 8192)
    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:   # ctypes releases the GIL
        want = list(ex.map(lambda s: PortOracle(**kw).run(iq[s]), range(n)))
    for s in range(n):
        assert np.array_equal(pcm[s], want[s]), f"stream {s}"


def test_oracle_on_this_box_still_matches_the_reference_golden_pcm():
    """The oracle libraries on the GPU box are the prebuilt ones: re-pin them here, in the -m gpu session too."""
    for cid, cfg, kind, stream, blocks in CASES:
        iq = make_input(cfg, kind, stream, blocks)
        assert sha(iq) == META["cases"][cid]["input_sha256"]
        assert np.array_equal(PortOracle(**CONFIGS[cfg]).run(iq), GOLD[cid]), cid


@pytest.mark.parametrize("segs", [1, 2, 4, 8])
@pytest.mark.parametrize("cfgname,kind", [("stereo192", "random"), ("mono192", "fm_mono"), ("stereo240", "random")])
def test_time_segmentation_does_not_change_the_result(cfgname, kind, segs):
    blocks = 6 if cfgname == "stereo240" else 2
    iq = np.stack([make_input(cfgname, kind, s, blocks) for s in range(2)])
    with R.FmBatch(cfg_for(cfgname, n_streams=2, segments=segs)) as fb:
        pcm = fb.run(iq)
    for s in range(2):
        assert np.array_equal(pcm[s], PortOracle(**CONFIGS[cfgname]).run(iq[s]))


@pytest.mark.parametrize("cfgname", ["mono240", "mono240_32", "mono240_off"])
def test_mono_off_the_4_to_1_path_runs_the_warp_specialised_kernel_and_equals_the_plain_one(monkeypatch, cfgname):
    """Mono ratios other than 4:1 (the reference's default 240 kHz among them) take the generic tick path of
    fmb_mono_ws_kernel; FMB_WS_GENERIC=0 sends them through fmb_demod_kernel.  Both against the oracle: a small batch
    (static split over the CTAs: runs that start inside a stream, with lead-ins) and ticketed whole-stream runs."""
    for n, blocks, ticketed in ((3, 3, False), (40, 2, True)):
        if ticketed:
            monkeypatch.setenv("FMB_CHUNK", "8"); monkeypatch.setenv("FMB_TAIL_PCT", "0")
        uniq = min(n, 3)
        iq = np.stack([make_input(cfgname, "fm_mono" if (s % uniq) % 2 else "random", s % uniq, blocks) for s in range(n)])
        want = [PortOracle(**CONFIGS[cfgname]).run(iq[s]) for s in range(uniq)]
        for generic, name in (("1", "fmb_mono_ws_kernel"), ("0", "fmb_demod_kernel")):
            monkeypatch.setenv("FMB_WS_GENERIC", generic)
            with R.FmBatch(cfg_for(cfgname, n_streams=n)) as fb:
                assert fb.kernel_name() == name
                pcm = fb.run(iq)
            for s in range(n):
                assert np.array_equal(pcm[s], want[s % uniq]), (cfgname, n, generic, s)


@pytest.mark.parametrize("cfgname,kind", [("stereo192", "fm_stereo"), ("stereo192", "random"), ("mono192", "random"),
                                          ("stereo240", "fm_stereo"), ("stereo170_44", "fm_stereo"),
                                          ("stereo170_44", "random"), ("mono240_32", "fm_mono"), ("mono240", "random")])
def test_fma_precision_within_one_lsb(cfgname, kind):
    blocks = 6 if cfgname in ("stereo240", "stereo170_44", "mono240_32", "mono240") else 3
    iq = make_input(cfgname, kind, 3, blocks)[None, :]
    with R.FmBatch(cfg_for(cfgname, n_streams=1, precision=R.FMB_PRECISION_FMA)) as fb:
        pcm = fb.run(iq)[0].astype(np.int32)
    want = PortOracle(**CONFIGS[cfgname]).run(iq[0]).astype(np.int32)
    assert pcm.shape == want.shape
    assert np.abs(pcm - want).max() <= 1      # tolerance: +-1 LSB of int16 PCM


def test_carried_state_equals_the_oracles_and_resumes_bit_exactly():
    """fmb_get_state mirrors the state fields of demod_state; a new handle restored from it
    continues bit-exactly (checkpoint/resume)."""
    cfgname = "stereo240"
    iq = np.stack([make_input(cfgname, "random", s, 5) for s in range(3)])
    orc = [PortOracle(**CONFIGS[cfgname]) for _ in range(3)]
    with R.FmBatch(cfg_for(cfgname, n_streams=3)) as fb:
        for b in range(3):
            fb.process(iq[:, b * B:(b + 1) * B])
            for s in range(3):
                orc[s].block(iq[s, b * B:(b + 1) * B])
        st, phase, blocks_done = fb.get_state()
        for s in range(3):
            o, oph, obl = orc[s].state()
            assert phase == oph and blocks_done == obl == 3
            for f, n in (("lowpass_tb", 48), ("br", 128), ("bm", 128), ("bs", 128)):
                of = "tb" if f == "lowpass_tb" else f
                assert same_floats(np.frombuffer(getattr(st[s], f), np.float32), np.frombuffer(getattr(o, of), np.float32)), (s, f)
            for f in ("pre_r", "pre_j", "pp", "deemph_l", "deemph_r"):
                assert np.float32(getattr(st[s], f)) == np.float32(getattr(o, f)), (s, f)
        rest = [fb.process(iq[:, b * B:(b + 1) * B]) for b in (3, 4)]
    with R.FmBatch(cfg_for(cfgname, n_streams=3)) as fb2:
        fb2.set_state(st, phase, blocks_done)
        rest2 = [fb2.process(iq[:, b * B:(b + 1) * B]) for b in (3, 4)]
    for a, b_ in zip(rest, rest2):
        assert np.array_equal(a, b_)
    for s in range(3):
        assert np.array_equal(rest[0][s], orc[s].block(iq[s, 3 * B:4 * B]))
        assert np.array_equal(rest[1][s], orc[s].block(iq[s, 4 * B:5 * B]))


def test_reset_restarts_the_stream():
    iq = make_input("stereo192", "random", 2, 2)[None, :]
    with R.FmBatch(cfg_for("stereo192", n_streams=1)) as fb:
        a = fb.run(iq)
        fb.reset()
        b = fb.run(iq)
    assert np.array_equal(a, b)


def test_three_host_paths_agree():
    """fmb_process, fmb_submit/fmb_wait (pipelined) and fmb_process_device give the same PCM."""
    import torch
    n, blocks = 5, 4
    iq = np.stack([make_input("stereo192", "fm_stereo", s, blocks) for s in range(n)])
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        ref = fb.run(iq)
    # pipelined, pinned
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        hin = [torch.from_numpy(iq[:, b * B:(b + 1) * B].copy()).pin_memory() for b in range(blocks)]
        hout = [torch.zeros((n, 8192), dtype=torch.int16).pin_memory() for _ in range(blocks)]
        tickets = []
        for b in range(blocks):
            if len(tickets) == L.FMB_PIPE_DEPTH:
                fb.wait(tickets.pop(0))
            tickets.append(fb.submit(hin[b].data_ptr(), B, hout[b].data_ptr(), 8192))
        for t in tickets:
            fb.wait(t)
        piped = np.concatenate([h.numpy() for h in hout], axis=1)
    assert np.array_equal(piped, ref)
    # device resident
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        d_in = torch.from_numpy(iq).cuda()
        d_out = torch.zeros((blocks, n, 8192), dtype=torch.int16, device="cuda")
        st = torch.cuda.current_stream().cuda_stream
        for b in range(blocks):
            fb.process_device(d_in.data_ptr() + b * B, iq.shape[1], d_out[b].data_ptr(), 8192, st)
        fb.join(st)
        torch.cuda.synchronize()
        dev = np.concatenate([d_out[b].cpu().numpy() for b in range(blocks)], axis=1)
    assert np.array_equal(dev, ref)


@pytest.mark.parametrize("n", [1, 31, 33, 97])
def test_ragged_stream_counts(n):
    iq = np.stack([make_input("stereo192", "random", s % 4, 1) for s in range(n)])
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        pcm = fb.run(iq)
    want = [PortOracle(**CONFIGS["stereo192"]).run(iq[s]) for s in range(min(n, 4))]
    for s in range(n):
        assert np.array_equal(pcm[s], want[s % 4])


def test_small_blocks_equal_one_reference_block():
    """block_bytes is any multiple of 32768; at 192 kHz (no in-place quirk) the split is invisible."""
    iq = make_input("stereo192", "random", 12, 2)[None, :]
    with R.FmBatch(cfg_for("stereo192", n_streams=1, block_bytes=32768)) as fb:
        small = fb.run(iq)
    assert np.array_equal(small[0], PortOracle(**CONFIGS["stereo192"]).run(iq[0]))


@pytest.mark.parametrize("offset", [0, 1])
def test_config_3_full_size_1024_streams(offset):
    """BASELINE.json configs[3]: 1024 streams, rotate and offset paths.  16 distinct channels are
    each checked against the oracle; the replicas must be identical to their originals."""
    n, uniq, blocks = 1024, 16, 2
    name = "stereo192_off" if offset else "stereo192"
    iq = R.synth.batch("fm_stereo", n, 192000, offset, blocks * B // 2, unique=uniq)
    with R.FmBatch(cfg_for(name, n_streams=n)) as fb:
        pcm = fb.run(iq)
    for s in range(uniq):
        assert np.array_equal(pcm[s], PortOracle(**CONFIGS[name]).run(iq[s])), s
    assert np.array_equal(pcm.reshape(n // uniq, uniq, -1), np.broadcast_to(pcm[:uniq], (n // uniq, uniq, pcm.shape[1])))


def test_config_4_maximum_size_8192_streams_on_one_gpu():
    """8192 streams (the whole configs[4] batch on ONE device, 2 GiB of IQ per step)."""
    n, uniq = 8192, 8
    iq = R.synth.batch("fm_stereo", n, 192000, 0, B // 2, unique=uniq)
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        pcm = fb.process(iq)
    for s in range(uniq):
        assert np.array_equal(pcm[s], PortOracle(**CONFIGS["stereo192"]).run(iq[s])), s
    sums = pcm.astype(np.int64).sum(axis=1).reshape(n // uniq, uniq)     # checksum of checksums
    assert (sums == sums[0]).all()


@pytest.mark.parametrize("cfgname,kind,chunk,tail", [("stereo192", "fm_stereo", 1, 100), ("stereo192", "random", 4, 50),
                                                     ("mono192", "fm_mono", 2, 100), ("mono192", "fm_mono", 8, 100),
                                                     ("stereo240", "fm_stereo", 2, 60), ("stereo192", "fm_stereo", 0, 0)])
def test_dynamic_work_assignment_does_not_change_the_result(monkeypatch, cfgname, kind, chunk, tail):
    """A batch that fills the GPU (>= SMs x resident CTAs work units) is handed out through the ticket
    counter: whole streams first, then chunks of `chunk` sub-tiles that re-enter a stream through the
    recomputed lead-in.  Every split must give the oracle's PCM, over several carried blocks."""
    monkeypatch.setenv("FMB_CHUNK", str(chunk))
    monkeypatch.setenv("FMB_TAIL_PCT", str(tail))
    n, uniq, blocks = 64, 8, 3
    c = CONFIGS[cfgname]
    iq = R.synth.batch(kind, n, c["rate_in"], c.get("offset_tuning", 0), blocks * B // 2, unique=uniq)
    with R.FmBatch(cfg_for(cfgname, n_streams=n)) as fb:
        pcm = fb.run(iq)
    for s in range(uniq):
        assert np.array_equal(pcm[s], PortOracle(**c).run(iq[s])), s
    assert np.array_equal(pcm.reshape(n // uniq, uniq, -1), np.broadcast_to(pcm[:uniq], (n // uniq, uniq, pcm.shape[1])))


def test_kernels_really_launch_and_errors_are_loud():
    iq = make_input("stereo192", "fm_stereo", 0, 1)[None, :]
    before = R.launch_count()
    with R.FmBatch(cfg_for("stereo192", n_streams=1)) as fb:
        fb.process(iq)
        assert R.launch_count() - before == 2           # demod + de-emphasis kernels
        pcm = np.zeros((1, 16), np.int16)
        rc = fb._lib.fmb_process(fb._h, iq.ctypes.data, B, pcm.ctypes.data, 16, None)
        assert rc == L.FMB_ERR_ARG                       # pcm_pitch < out count
        assert fb._lib.fmb_wait(fb._h, 12345, None) == L.FMB_ERR_STATE


def test_inplace_hazard_is_refused_at_create_not_in_the_middle_of_playback():
    """A stereo rate ratio between 2 and 3 whose block-start phases reach a tick on sample <= 2 would make the
    reference's in-place output overwrite unread input beyond the emulated first-sample case (:593-597).
    100000/48000 does so on its third block (phase 64000): refused by fmb_create, and by fmb_set_state for an
    imported phase -- never silently wrong, never an abort after two good blocks."""
    for name, kw in REFUSED.items():
        with pytest.raises(R.FmbError) as e:
            R.FmBatch(R.DemodConfig(n_streams=1, **kw))
        assert e.value.code == L.FMB_ERR_UNSUPPORTED, name
    # ratio 2.67: 16384*48000 is a multiple of 128000, every block starts at phase 0: fine; an imported phase of
    # 120000 >= 2*128000 - 3*48000 puts tick 1 on sample 2: refused
    kw = dict(CONFIGS["stereo192"], rate_in=128000)
    iq = make_input("stereo192", "random", 1, 2)
    with R.FmBatch(R.DemodConfig(n_streams=1, **kw)) as fb:
        pcm = fb.run(iq[None, :])
        assert np.array_equal(pcm[0], PortOracle(**kw).run(iq))
        st, _, _ = fb.get_state()
        with pytest.raises(R.FmbError) as e:
            fb.set_state(st, 120000, 0)
        assert e.value.code == L.FMB_ERR_UNSUPPORTED


def test_caller_may_alternate_cuda_streams_between_steps():
    """fmb_process_device on a different stream than the previous step first waits (device side) for that
    step's demodulation: the carried state ping-pongs between the two calls.  Alternating two streams, with no
    host synchronisation in between, must still give the oracle's PCM."""
    import torch
    n, blocks = 96, 6
    uniq = 4
    iq = np.stack([make_input("stereo192", "fm_stereo", s % uniq, blocks) for s in range(n)])
    want = [PortOracle(**CONFIGS["stereo192"]).run(iq[s]) for s in range(uniq)]
    d_in = torch.from_numpy(iq).cuda()
    d_out = torch.zeros((blocks, n, 8192), dtype=torch.int16, device="cuda")
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        for b in range(blocks):
            fb.process_device(d_in.data_ptr() + b * B, iq.shape[1], d_out[b].data_ptr(), 8192, streams[b & 1].cuda_stream)
        for st in streams:
            fb.join(st.cuda_stream)
        torch.cuda.synchronize()
    got = np.concatenate([d_out[b].cpu().numpy() for b in range(blocks)], axis=1)
    for s in range(n):
        assert np.array_equal(got[s], want[s % uniq]), s


def test_rate_out_below_rate_in_follows_the_reference():
    """-o 2 configurations (filters at rate_in, ticks at rate_out) across carried blocks, several channels."""
    for name, kind in (("stereo384_o2", "random"), ("stereo480_o2", "fm_stereo"), ("mono384_o2", "random")):
        kw = CONFIGS[name]
        blocks = 6 if name == "stereo480_o2" else 2
        iq = np.stack([make_input(name, kind, s, blocks) for s in range(3)])
        with R.FmBatch(cfg_for(name, n_streams=3)) as fb:
            pcm = fb.run(iq)
        for s in range(3):
            assert np.array_equal(pcm[s], PortOracle(**kw).run(iq[s])), (name, s)


def test_deemphasis_speculation_is_verified_and_falls_back_on_digital_silence():
    """Kernel 2 runs the IIR speculatively in time and verifies every junction.  On a real FM
    signal in steady state the verification passes (no sequential redo); on constant bytes the
    true state sticks at a denormal, the speculation fails, every chunk is redone in order --
    and the PCM is the oracle's in both cases."""
    blocks = 4
    for kind in ("fm_stereo", "const127"):
        iq = make_input("stereo192", kind, 0, blocks)[None, :]
        orc = PortOracle(**CONFIGS["stereo192"])
        with R.FmBatch(cfg_for("stereo192", n_streams=1)) as fb:
            counts = []
            for b in range(blocks):
                pcm = fb.process(iq[:, b * B:(b + 1) * B])
                assert np.array_equal(pcm[0], orc.block(iq[0, b * B:(b + 1) * B]))
                counts.append(fb.deemph_fallbacks())
        if kind == "fm_stereo":
            assert counts[-1] == counts[0] <= 2, counts      # at most the start-up transient
        else:
            assert counts[-1] >= 8 * (blocks - 1), counts    # 8 chunks of 1024 values per block


@pytest.mark.parametrize("pitch_extra", [0, 1, 3, 8])
def test_unaligned_pcm_pitch(pitch_extra):
    """PCM rows that are not 16-byte aligned take the scalar store path."""
    n = 3
    iq = np.stack([make_input("stereo240", "random", s, 2) for s in range(n)])
    want = [PortOracle(**CONFIGS["stereo240"]).run(iq[s]) for s in range(n)]
    with R.FmBatch(cfg_for("stereo240", n_streams=n)) as fb:
        got = []
        for b in range(2):
            cnt = fb.next_out_count()
            pitch = cnt + pitch_extra
            pcm = np.zeros((n, pitch), np.int16)
            blk = np.ascontiguousarray(iq[:, b * B:(b + 1) * B])
            L.check(fb._lib.fmb_process(fb._h, blk.ctypes.data, B, pcm.ctypes.data, pitch, None), "fmb_process")
            got.append(pcm[:, :cnt])
    got = np.concatenate(got, axis=1)
    for s in range(n):
        assert np.array_equal(got[s], want[s])


def test_whole_stream_runs_on_random_bytes(monkeypatch):
    """Dynamic assignment, every stream handed out whole (8 consecutive sub-tiles per CTA, the carried
    sub-tile state chained through shared memory), on uniform-random bytes (every atan2 branch)."""
    monkeypatch.setenv("FMB_CHUNK", "8")
    monkeypatch.setenv("FMB_TAIL_PCT", "0")
    n, uniq, blocks = 64, 4, 2
    iq = np.stack([make_input("stereo192", "random", s % uniq, blocks) for s in range(n)])
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb:
        pcm = fb.run(iq)
    want = [PortOracle(**CONFIGS["stereo192"]).run(iq[s]) for s in range(uniq)]
    for s in range(n):
        assert np.array_equal(pcm[s], want[s % uniq]), s


@pytest.mark.parametrize("cfgname,kind", [("stereo192", "fm_stereo"), ("mono192", "fm_mono"), ("stereo240", "random"),
                                          ("mono240", "fm_mono")])
@pytest.mark.parametrize("pdl", ["1", "0"])
def test_back_to_back_launches_of_a_full_batch_overlap_and_stay_exact(monkeypatch, cfgname, kind, pdl):
    """1024 streams x 6 blocks enqueued back to back on one stream, no host synchronisation in between: consecutive
    demod launches overlap at their ends (programmatic dependent launch; FMB_PDL=0: plain stream order), every stream
    is handed out whole through the ticket counter, the carried state and the decoder-output buffers are ordered per
    stream inside the kernels.  mono192 runs the warp-specialised kernel, stereo240 the in-place quirk, mono240 the
    generic tick path.  16 distinct channels against the oracle, every replica identical to its original."""
    run_back_to_back(monkeypatch, cfgname, kind, pdl)


def run_back_to_back(monkeypatch, cfgname, kind, pdl, fma=False):
    """fma: FMB_PRECISION_FMA against the fused restatement."""
    import torch
    monkeypatch.setenv("FMB_PDL", pdl)
    n, uniq, blocks = 1024, 16, 6
    c = CONFIGS[cfgname]
    precision = R.FMB_PRECISION_FMA if fma else R.FMB_PRECISION_EXACT
    iq_u = np.stack([make_input(cfgname, kind, s, blocks) for s in range(uniq)])
    d_u = torch.from_numpy(iq_u).cuda()
    idx = torch.arange(n, device="cuda") % uniq
    d_in = [d_u[:, b * B:(b + 1) * B].index_select(0, idx).contiguous() for b in range(blocks)]
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    with R.FmBatch(cfg_for(cfgname, n_streams=n, precision=precision)) as fb:
        pitch = (fb.max_out + 7) & ~7
        d_out = torch.zeros((blocks, n, pitch), dtype=torch.int16, device="cuda")
        counts = []
        torch.cuda.synchronize()
        for b in range(blocks):
            counts.append(fb.next_out_count())
            fb.process_device(d_in[b].data_ptr(), B, d_out[b].data_ptr(), pitch, st.cuda_stream)
        fb.join(st.cuda_stream)
        torch.cuda.synchronize()
        fb.get_state(0, 1)                               # reports a device-side hand-over time-out, if any
    got = np.concatenate([d_out[b, :, :counts[b]].cpu().numpy() for b in range(blocks)], axis=1)
    for s in range(uniq):
        assert np.array_equal(got[s], PortOracle(**c, fma=fma).run(iq_u[s])), s
    assert np.array_equal(got.reshape(n // uniq, uniq, -1), np.broadcast_to(got[:uniq], (n // uniq, uniq, got.shape[1])))


def test_iq_produced_by_a_kernel_on_the_same_stream_right_before_the_step():
    """Consecutive demod launches overlap, so a launch does not wait for the complete end of a KERNEL enqueued on
    its stream immediately before it (fmb.h, "Input readiness").  A caller whose own kernel produces the IQ says so
    with fmb_input_ready(): here every block is copied into the input buffer by a device kernel on the same stream
    right before the step, with no host synchronisation anywhere."""
    import torch
    n, uniq, blocks = 1024, 8, 5
    iq_u = np.stack([make_input("stereo192", "fm_stereo", s, blocks) for s in range(uniq)])
    d_u = torch.from_numpy(iq_u).cuda()
    idx = torch.arange(n, device="cuda") % uniq
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    with R.FmBatch(cfg_for("stereo192", n_streams=n)) as fb, torch.cuda.stream(st):
        d_in = [torch.empty((n, B), dtype=torch.uint8, device="cuda") for _ in range(2)]
        d_out = torch.zeros((blocks, n, 8192), dtype=torch.int16, device="cuda")
        for b in range(blocks):
            torch.index_select(d_u[:, b * B:(b + 1) * B], 0, idx, out=d_in[b & 1])     # a kernel on `st` writes the IQ ...
            fb.input_ready()                                                            # ... so say so
            fb.process_device(d_in[b & 1].data_ptr(), B, d_out[b].data_ptr(), 8192, st.cuda_stream)
        fb.join(st.cuda_stream)
    torch.cuda.synchronize()
    got = np.concatenate([d_out[b].cpu().numpy() for b in range(blocks)], axis=1)
    for s in range(uniq):
        assert np.array_equal(got[s], PortOracle(**CONFIGS["stereo192"]).run(iq_u[s])), s
    assert np.array_equal(got.reshape(n // uniq, uniq, -1), np.broadcast_to(got[:uniq], (n // uniq, uniq, got.shape[1])))
