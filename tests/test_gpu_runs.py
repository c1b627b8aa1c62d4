"""Several consecutive blocks of every stream in one call (fmb_config.max_blocks_per_call, fmb_set_blocks_per_call).

A call of n blocks must be bit for bit what n one-block calls produce: PCM, out counts, the discriminator and decoder
taps, the carried state, the resampler phase and the block counter, in both precisions and for every configuration.
Everything here is compared with the C restatement (PortOracle) run block by block.  The call sequences change n
between calls, so the in-place quirk (SURVEY A.7) falls at block starts inside a call's row, and the work assignment
and the de-emphasis time segments change from call to call."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from oracle.oracle_py import PortOracle
from rtl_fm_player_b200 import _lib as L
from vectors import B, CONFIGS, LONG_CASES, long_capture_bytes, make_input, sha

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SEQ = [1, 3, 8, 2, 7]
ALL = ["stereo192", "stereo240", "stereo480_o2", "stereo170_44", "stereo192_128", "stereo192_off", "mono192", "mono240",
       "mono240_32", "drop192", "nolpr192", "nodeemph192"]


def fast_of(kw):
    return kw.get("rate_out") or kw["rate_in"]


def kind_of(kw):
    return "fm_stereo" if kw["mode"] == 2 else "fm_mono"


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def quirk_phase(kw, phase):
    return kw["mode"] == 2 and kw["rate_out2"] > 0 and phase + kw["rate_out2"] >= fast_of(kw)


def check_state(fb, orcs, rows, kw, where):
    gst, phase, done = fb.get_state()
    for s, o in enumerate(orcs):
        ost, ophase, odone = o.state()
        assert (phase, done) == (ophase, odone), f"{where}: phase / block counter"
        g = gst[list(rows).index(s)]
        names = ["lowpass_tb", "pre_r", "pre_j", "deemph_l"]
        if kw["rate_out2"] > 0:                      # without lp_real_f32 the restatement keeps no lpr.br ring
            names.append("br")
        if kw["mode"] == 2 and kw["rate_out2"] > 0:
            names += ["bm", "bs", "pp", "deemph_r"]
        for f in names:
            gf = np.array(getattr(g, f), dtype=np.float32, ndmin=1)
            of = np.array(getattr(ost, "tb" if f == "lowpass_tb" else f), dtype=np.float32, ndmin=1)
            assert np.array_equal(bits(gf), bits(of)), f"{where}: carried {f} differs"


def run_calls(kw, seq, n_streams=2, uniq=None, bb=B, fma=False, taps=True, kind=None, iq=None, **extra):
    """Calls of seq[i] blocks on one handle against the oracle run block by block (stream s = unique row s % uniq).
    Returns (handle's concatenated PCM of row 0, the block-start phases that carried the quirk inside a call)."""
    uniq = uniq or min(n_streams, 3)
    total = sum(seq)
    if iq is None:
        iq = np.stack([R.synth.capture(kind or kind_of(kw), s, kw["rate_in"], kw.get("offset_tuning", 0), total * bb // 2)
                       for s in range(uniq)])
    rows = np.arange(n_streams) % uniq
    orcs = [PortOracle(**kw, fma=fma) for _ in range(uniq)]
    inner_quirks = 0
    got = []
    cfg = R.DemodConfig(**kw, n_streams=n_streams, block_bytes=bb, max_blocks_per_call=max(seq),
                        precision=R.FMB_PRECISION_FMA if fma else R.FMB_PRECISION_EXACT, **extra)
    with R.FmBatch(cfg) as fb:
        if taps:
            fb.debug_enable(True)
        off = 0
        for n in seq:
            fb.set_blocks_per_call(n)
            phase = fb.get_state(0, 1)[1]
            want_counts = [fb.out_count_blocks(j) for j in range(n + 1)]
            assert want_counts[n] == fb.next_out_count()
            per = [[o.block(iq[s, (off + b) * bb:(off + b + 1) * bb], stages=True) for b in range(n)]
                   for s, o in enumerate(orcs)]
            for b in range(1, n):
                p = (phase + b * (bb // 16) * kw["rate_out2"]) % fast_of(kw) if kw["rate_out2"] > 0 else 0
                inner_quirks += quirk_phase(kw, p)
            batch = np.ascontiguousarray(iq[rows, off * bb:(off + n) * bb])
            pcm = fb.process(batch)
            for s in range(uniq):
                want = np.concatenate([pb[0] for pb in per[s]])
                assert [0] + list(np.cumsum([len(pb[0]) for pb in per[s]])) == want_counts, "out counts"
                for r in np.nonzero(rows == s)[0]:
                    assert np.array_equal(pcm[r], want), f"call of {n} blocks at block {off}, stream {r}: PCM"
            if taps:
                dem, lr = fb.debug_read()
                for s in range(uniq):
                    r = int(np.nonzero(rows == s)[0][0])
                    assert np.array_equal(bits(dem[r]), bits(np.concatenate([pb[1]["dem"] for pb in per[s]]))), \
                        f"call of {n} blocks at block {off}: discriminator tap"
                    wl = np.concatenate([pb[1]["lr"] for pb in per[s]])
                    assert np.array_equal(bits(lr[r, :len(wl)]), bits(wl)), f"call of {n} blocks at block {off}: decoder tap"
            check_state(fb, orcs, rows, kw, f"after the call of {n} blocks at block {off}")
            got.append(pcm[0])
            off += n
    return np.concatenate(got), inner_quirks


@pytest.mark.parametrize("name", ALL)
def test_changing_blocks_per_call_equals_block_by_block(name):
    _, q = run_calls(CONFIGS[name], SEQ)
    if name in ("stereo240", "stereo480_o2"):
        assert q > 0, "the quirk must fall on block starts inside calls"


@pytest.mark.parametrize("name", ["stereo240", "stereo192", "mono240"])
def test_fma_changing_blocks_per_call_equals_the_fused_restatement(name):
    run_calls(CONFIGS[name], SEQ, fma=True)


@pytest.mark.parametrize("name,bb,seq", [("stereo240", 32768, [1, 40, 7, 13]), ("stereo240", 98304, [5, 40, 2]),
                                         ("stereo170_44", 32768, [40, 3]), ("mono240", 98304, [40, 1, 9]),
                                         ("stereo192", 32768, [17, 40])])
def test_small_blocks_put_block_starts_at_every_sub_tile(name, bb, seq):
    """32 768-byte blocks start at every sub-tile; 98 304-byte blocks off the 8-sub-tile grid."""
    run_calls(CONFIGS[name], seq, bb=bb, n_streams=1)


def phases_to_test(kw, sample=None, seed=3):
    import math
    fast, step = fast_of(kw), (B // 16) * kw["rate_out2"] % fast_of(kw)
    n = fast // math.gcd(step, fast)
    cyc = [(k * step) % fast for k in range(n)]
    if sample and len(cyc) > sample:
        import random
        cyc = sorted(set(cyc[:4] + random.Random(seed).sample(cyc, sample)))
    return cyc


@pytest.mark.parametrize("name,sample", [("stereo240", None), ("stereo480_o2", None), ("stereo170_44", 24)])
@pytest.mark.parametrize("raw_valid", [0, 1])
def test_every_block_start_phase_then_one_multi_block_call(name, sample, raw_valid):
    """The handle and the oracle are put into the same state at each block-start phase of the cycle (fmb_set_state,
    raw_valid 0: from the oracle's floats; 1: the handle's own exported state), then one call of 6 blocks."""
    kw = CONFIGS[name]
    n = 6
    iq = R.synth.capture("fm_stereo", 1, kw["rate_in"], kw.get("offset_tuning", 0), (n + 1) * B // 2)
    with R.FmBatch(R.DemodConfig(**kw, n_streams=1, max_blocks_per_call=n)) as fb:
        fb.set_blocks_per_call(1)
        orc = PortOracle(**kw)
        fb.process(iq[None, :B])
        orc.block(iq[:B])
        base, _, _ = fb.get_state()
        obase = orc.state()[0]
        for p in phases_to_test(kw, sample):
            st = (L.FmbStreamState * 1)()
            if raw_valid:
                C.memmove(C.addressof(st[0]), C.addressof(base[0]), C.sizeof(L.FmbStreamState))
            else:
                C.memmove(C.addressof(st[0]), C.addressof(obase), L.FmbStreamState.raw_valid.offset)
                st[0].raw_valid = 0
            fb.set_state(st, p, 1)
            o = PortOracle(**kw)
            o.set_state(obase, p, 1)
            fb.set_blocks_per_call(n)
            pcm = fb.process(iq[None, B:])
            want = np.concatenate([o.block(iq[(b + 1) * B:(b + 2) * B]) for b in range(n)])
            assert np.array_equal(pcm[0], want), f"phase {p}"
            check_state(fb, [o], [0], kw, f"phase {p}")


@pytest.mark.parametrize("name,n_streams,seq,env", [
    ("stereo240", 1, [64], {}),                               # 512 units on 444 CTAs: static split, lead-ins
    ("stereo192", 1, [64, 3], {}),
    ("mono240", 1, [64], {}),
    ("stereo240", 31, [5, 2, 8], {}),
    ("stereo240", 1024, [2, 1, 2], {}),                       # tickets of one block each
    ("stereo192", 1024, [2, 2], {}),
    ("mono192", 1024, [2, 1], {}),
    ("stereo240", 96, [4, 3], {"FMB_CHUNK": "2", "FMB_TAIL_PCT": "50"}),
    ("stereo240", 96, [4, 3], {"FMB_CHUNK": "0"}),
    ("stereo240", 8, [3, 2, 4], {"segments": 4}),
    ("stereo170_44", 8, [2, 5], {"segments": 2}),
    ("stereo240", 1024, [2, 2, 2], {"FMB_PDL": "0"}),
    ("stereo240", 1024, [2, 2, 2], {"FMB_PDL": "1"}),
    ("mono240", 4, [6, 2], {"FMB_WS": "0"}),
    ("mono192", 4, [6, 2], {"FMB_WS": "0"}),
])
def test_work_assignment_regimes(monkeypatch, name, n_streams, seq, env):
    extra = {}
    for k, v in env.items():
        if k == "segments":
            extra["segments"] = v
        else:
            monkeypatch.setenv(k, v)
    run_calls(CONFIGS[name], seq, n_streams=n_streams, uniq=min(n_streams, 4), taps=n_streams <= 32, **extra)


def test_deemphasis_segments_pole_close_to_one():
    """A pole close to 1 (20 ms): the speculation of every time segment converges late or not at all."""
    kw = dict(CONFIGS["stereo192"], deemph=0.020)
    run_calls(kw, [64, 1, 20], n_streams=1)


def test_deemphasis_segments_repair_every_junction_on_silence():
    """Digital silence over 64 blocks: the true state sticks at a denormal while every speculating segment stays at 0,
    so every junction is repaired in order -- and the counter of redone chunks rises by at least the row's length."""
    kw = CONFIGS["stereo192"]
    iq = R.synth.capture("const127", 0, kw["rate_in"], 0, 64 * B // 2)[None, :]
    orc = PortOracle(**kw)
    with R.FmBatch(R.DemodConfig(**kw, n_streams=1, max_blocks_per_call=64)) as fb:
        f0 = fb.deemph_fallbacks()
        pcm = fb.process(iq)
        f1 = fb.deemph_fallbacks()
    want = np.concatenate([orc.block(iq[0, b * B:(b + 1) * B]) for b in range(64)])
    assert np.array_equal(pcm[0], want)
    assert f1 - f0 >= 7 * 64, (f0, f1)


def test_deemphasis_off_over_long_rows():
    run_calls(CONFIGS["nodeemph192"], [64, 2], n_streams=1)


@pytest.mark.parametrize("case", LONG_CASES, ids=[c[0] for c in LONG_CASES])
def test_ten_second_captures_in_calls_of_64(case):
    import json
    meta = json.load(open(os.path.join(HERE, "golden", "golden_meta.json")))["long"]
    cid, cfg, kind, stream, blocks = case
    iq = make_input(cfg, kind, stream, blocks)
    with R.FmBatch(R.DemodConfig(**CONFIGS[cfg], n_streams=1, max_blocks_per_call=64)) as fb:
        pcm = fb.run(np.concatenate([iq, np.zeros(long_capture_bytes(cfg) - blocks * B, np.uint8)])[None, :])
    assert pcm.shape[1] == meta[cid]["n_pcm"] and sha(pcm[0]) == meta[cid]["pcm_sha256"]


def test_pipelined_submits_remember_their_own_block_count():
    kw = CONFIGS["stereo240"]
    n_streams, seq = 3, [4, 1, 6]
    iq = np.stack([R.synth.capture("fm_stereo", s, kw["rate_in"], 0, sum(seq) * B // 2) for s in range(n_streams)])
    orcs = [PortOracle(**kw) for _ in range(n_streams)]
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n_streams, max_blocks_per_call=6)) as fb:
        pitch = (fb.max_out + 7) & ~7
        bufs, tickets, counts, off = [], [], [], 0
        for n in seq:
            fb.set_blocks_per_call(n)
            counts.append(fb.next_out_count())
            src = np.ascontiguousarray(iq[:, off * B:(off + n) * B])
            dst = np.zeros((n_streams, pitch), np.int16)
            bufs.append((src, dst))
            tickets.append(fb.submit(src.ctypes.data, src.strides[0], dst.ctypes.data, pitch))
            off += n
        for t, cnt, (src, dst), n in zip(tickets, counts, bufs, seq):
            n_out = (C.c_int * n_streams)()
            L.check(R.lib().fmb_wait(fb._h, t, n_out), "fmb_wait")
            assert list(n_out) == [cnt] * n_streams
        off = 0
        for (src, dst), n, cnt in zip(bufs, seq, counts):
            for s in range(n_streams):
                want = np.concatenate([orcs[s].block(iq[s, (off + b) * B:(off + b + 1) * B]) for b in range(n)])
                assert np.array_equal(dst[s, :cnt], want)
            off += n
        assert fb.get_state()[2] == sum(seq)


def test_device_resident_calls_on_a_caller_stream():
    import torch
    kw = CONFIGS["stereo240"]
    n_streams, seq = 4, [5, 2, 5]
    iq = np.stack([R.synth.capture("fm_stereo", s, kw["rate_in"], 0, sum(seq) * B // 2) for s in range(n_streams)])
    orcs = [PortOracle(**kw) for _ in range(n_streams)]
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n_streams, max_blocks_per_call=5)) as fb:
        s = torch.cuda.Stream()
        pitch = (fb.max_out + 7) & ~7
        off = 0
        for n in seq:
            fb.set_blocks_per_call(n)
            cnt = fb.next_out_count()
            with torch.cuda.stream(s):
                d_iq = torch.from_numpy(np.ascontiguousarray(iq[:, off * B:(off + n) * B])).cuda(non_blocking=False)
                d_iq = d_iq + 0                                 # produced by a kernel right before the step
                d_pcm = torch.zeros((n_streams, pitch), dtype=torch.int16, device="cuda")
            fb.input_ready()
            fb.process_device(d_iq.data_ptr(), n * B, d_pcm.data_ptr(), pitch, s.cuda_stream)
            fb.join(s.cuda_stream)
            s.synchronize()
            pcm = d_pcm.cpu().numpy()
            for r in range(n_streams):
                want = np.concatenate([orcs[r].block(iq[r, (off + b) * B:(off + b + 1) * B]) for b in range(n)])
                assert np.array_equal(pcm[r, :cnt], want)
            off += n


@pytest.mark.parametrize("shared", [False, True])
def test_multi_gpu_host_with_several_blocks_per_call(shared):
    kw = CONFIGS["stereo240"]
    n_dev = R.device_count()
    devices = [0, 0] if shared or n_dev < 2 else list(range(n_dev))
    n_streams = 2 * len(devices)
    seq = [3, 1, 4]
    iq = np.stack([R.synth.capture("fm_stereo", s % 3, kw["rate_in"], 0, sum(seq) * B // 2) for s in range(n_streams)])
    orcs = [PortOracle(**kw) for _ in range(3)]
    want = [orcs[s].run(iq[s]) for s in range(3)]
    with R.FmMulti(R.DemodConfig(**kw, n_streams=n_streams, max_blocks_per_call=4), devices) as fm:
        got, off = [], 0
        for n in seq:
            stage = R.pinned_array((n_streams, n * B), np.uint8)
            stage[...] = iq[:, off * B:(off + n) * B]
            fm.set_blocks_per_call(n)
            assert fm.out_count_blocks(n) == fm.next_out_count()
            got.append(fm.process(stage).copy())
            R.free_pinned(stage)
            off += n
    pcm = np.concatenate(got, axis=1)
    for s in range(n_streams):
        assert np.array_equal(pcm[s], want[s % 3]), f"stream {s}"


def test_player_with_several_blocks_per_step_writes_the_same_files(tmp_path):
    """fmb_player -K 8 against -K 1 on three captures of different lengths, none a multiple of 8 blocks."""
    player = os.path.join(ROOT, "rtl_fm_player_b200", "fmb_player")
    files = []
    for i, blocks in enumerate([13, 21, 6]):
        p = tmp_path / f"cap{i}.u8"
        make_input("stereo192", "fm_stereo", i, blocks).tofile(p)
        files.append(str(p))
    outs = {}
    for K in (1, 8):
        for fmt in ("-w", None):
            d = tmp_path / f"out_K{K}_{fmt}"
            d.mkdir()
            cmd = [player, "-X", "-o", str(d), "-K", str(K)] + ([fmt] if fmt else []) + files
            r = subprocess.run(cmd, capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            outs[(K, fmt)] = {f.name: f.read_bytes() for f in sorted(d.iterdir())}
    for fmt in ("-w", None):
        assert outs[(1, fmt)].keys() == outs[(8, fmt)].keys() and len(outs[(1, fmt)]) == 3
        for k in outs[(1, fmt)]:
            assert outs[(1, fmt)][k] == outs[(8, fmt)][k], k
    kw = CONFIGS["stereo192"]
    for i, blocks in enumerate([13, 21, 6]):
        pcm = np.frombuffer(outs[(8, None)][f"cap{i}.u8.pcm"], dtype=np.int16)
        assert np.array_equal(pcm, PortOracle(**kw).run(make_input("stereo192", "fm_stereo", i, blocks)))


def test_defaults_and_arguments_on_a_handle():
    kw = CONFIGS["stereo240"]
    with R.FmBatch(R.DemodConfig(**kw)) as fb:               # no maximum: one block per call, as before
        with pytest.raises(R.FmbError):
            fb.set_blocks_per_call(2)
        assert fb.out_count_blocks(1) == fb.next_out_count()
    with R.FmBatch(R.DemodConfig(**kw, max_blocks_per_call=5)) as fb:
        assert fb.next_out_count() == fb.out_count_blocks(5)  # the default is the maximum
        one = R.FmBatch(R.DemodConfig(**kw))
        assert fb.max_out >= 5 * one.max_out - 2 and fb.max_out <= 5 * one.max_out
        one.close()
        for bad in (0, 6, -1):
            with pytest.raises(R.FmbError) as e:
                fb.set_blocks_per_call(bad)
            assert e.value.code == L.FMB_ERR_ARG
        fb.set_blocks_per_call(2)
        fb.reset()
        assert fb.next_out_count() == fb.out_count_blocks(2)  # reset keeps it


@pytest.mark.parametrize("name,n_streams,n", [("mono192", 8, 16), ("mono192", 1, 64), ("stereo192", 8, 16),
                                              ("mono240", 64, 4)])
def test_back_to_back_multi_block_calls_without_a_host_sync(name, n_streams, n):
    """Six device-resident calls enqueued back to back: a segmented de-emphasis pass is as long as such a demod launch,
    and the launches that reuse its decoder-output buffer must not wait for it inside the kernel (a hand-over wait
    once timed out here).  Every call's PCM against the oracle."""
    import torch
    kw = CONFIGS[name]
    calls, uniq = 6, 2
    iq = np.stack([R.synth.capture(kind_of(kw), s, kw["rate_in"], 0, calls * n * B // 2) for s in range(uniq)])
    rows = np.arange(n_streams) % uniq
    orcs = [PortOracle(**kw) for _ in range(uniq)]
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n_streams, max_blocks_per_call=n)) as fb:
        pitch = (fb.max_out + 7) & ~7
        st = R.lib().fmb_internal_stream(fb._h)
        d_iq = torch.from_numpy(np.ascontiguousarray(iq[rows])).cuda()
        torch.cuda.synchronize()
        outs, counts = [], []
        for k in range(calls):
            counts.append(fb.next_out_count())
            outs.append(torch.zeros((n_streams, pitch), dtype=torch.int16, device="cuda"))
            fb.process_device(d_iq.data_ptr() + k * n * B, calls * n * B, outs[-1].data_ptr(), pitch, st)
        L.check(R.lib().fmb_sync(fb._h), "fmb_sync")
        for k in range(calls):
            pcm = outs[k].cpu().numpy()
            for s in range(uniq):
                want = np.concatenate([orcs[s].block(iq[s, (k * n + b) * B:(k * n + b + 1) * B]) for b in range(n)])
                for r in np.nonzero(rows == s)[0]:
                    assert np.array_equal(pcm[r, :counts[k]], want), f"call {k}, stream {r}"
