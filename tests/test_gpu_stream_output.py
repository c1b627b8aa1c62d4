"""Per-stream output settings (fmb_set_stream_output): volume, de-emphasis time constant and pole for every stream of a
batch, changeable between calls.

Stream s of a mixed batch must be bit for bit what the C restatement (PortOracle) produces with s's settings: PCM, out
counts and the de-emphasis memories, with the discriminator and decoder taps those of the restatement (the settings
only act after the decoder).  The settings cycle through 50 us, 75 us, off and a pole near 1 (a time constant of 1 s),
and volumes 0, 0.4, -1.5 and 40 (saturating)."""
import os
import subprocess

import numpy as np
import pytest

import rtl_fm_player_b200 as R
from oracle.oracle_py import PortOracle
from rtl_fm_player_b200 import _lib as L
from vectors import B, CONFIGS

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEEMPH = [0.000050, 0.000075, 0.0, 1.0]
VOLUME = [0.0, 0.4, -1.5, 40.0]
P = 8                                   # setting classes: stream s has class s % P


def setting(k):
    """(deemph, volume) of class k: every deemph meets every volume class over the 8 classes."""
    k %= P
    return DEEMPH[k % 4], VOLUME[(k + k // 4) % 4]


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def kind_of(kw):
    return "fm_stereo" if kw["mode"] == 2 else "fm_mono"


def stereo_out(kw):
    return kw["mode"] == 2 and kw["rate_out2"] > 0


def oracle(kw, deemph, volume, fma=False):
    return PortOracle(**{**kw, "deemph": deemph, "volume": volume}, fma=fma)


def captures(kw, n, blocks, bb=B):
    return np.stack([R.synth.capture(kind_of(kw), s, kw["rate_in"], kw.get("offset_tuning", 0), blocks * bb // 2)
                     for s in range(n)])


def check_de_state(fb, orcs, rows, kw, where):
    gst = fb.get_state()[0]
    names = ["deemph_l"] + (["deemph_r"] if stereo_out(kw) else [])
    for u, o in enumerate(orcs):
        ost = o.state()[0]
        for r in np.nonzero(rows == u)[0][:4]:
            for f in names:
                assert bits(getattr(gst[int(r)], f)) == bits(getattr(ost, f)), f"{where}, stream {r}: {f}"


def run_mixed(kw, n_streams, seq=(1, 1), fma=False, shift=0, taps=None):
    """Calls of seq[i] blocks on a handle whose stream s carries setting(s + shift), against one restatement per class
    (input row s % P).  Returns the handle's de-emphasis fallback count."""
    uniq = min(n_streams, P)
    iq = captures(kw, uniq, sum(seq))
    rows = np.arange(n_streams) % uniq
    orcs = [oracle(kw, *setting(u + shift), fma=fma) for u in range(uniq)]
    taps = n_streams <= P if taps is None else taps
    cfg = R.DemodConfig(**kw, n_streams=n_streams, max_blocks_per_call=max(seq),
                        precision=R.FMB_PRECISION_FMA if fma else R.FMB_PRECISION_EXACT)
    d, v = zip(*(setting(s + shift) for s in range(n_streams)))
    with R.FmBatch(cfg) as fb:
        assert fb.deemph_kernel_name() in ("fmb_deemph_kernel", "fmb_deemph_seg_kernel")
        fb.set_stream_output(volume=np.array(v), deemph=np.array(d))
        so = fb.stream_output()
        assert np.array_equal(so["volume"], np.array(v, np.float32))
        assert np.array_equal(so["deemph_on"], np.array(d) != 0)
        if taps:
            fb.debug_enable(True)
        off = 0
        for n in seq:
            fb.set_blocks_per_call(n)
            name = fb.deemph_kernel_name()
            assert name.endswith("_per_stream") and (("seg" in name) == (n > 1 and n_streams < 64)), name
            per = [[o.block(iq[u, (off + b) * B:(off + b + 1) * B], stages=True) for b in range(n)]
                   for u, o in enumerate(orcs)]
            pcm = fb.process(np.ascontiguousarray(iq[rows, off * B:(off + n) * B]))
            for u in range(uniq):
                want = np.concatenate([pb[0] for pb in per[u]])
                assert pcm.shape[1] == len(want), "out count"
                for r in np.nonzero(rows == u)[0]:
                    assert np.array_equal(pcm[r], want), f"call of {n} at block {off}, stream {r} {setting(r + shift)}"
            if taps:
                dem, lr = fb.debug_read()
                for u in range(uniq):
                    wl = np.concatenate([pb[1]["lr"] for pb in per[u]])
                    assert np.array_equal(bits(dem[u]), bits(np.concatenate([pb[1]["dem"] for pb in per[u]])))
                    assert np.array_equal(bits(lr[u, :len(wl)]), bits(wl))
            check_de_state(fb, orcs, rows, kw, f"after the call at block {off}")
            off += n
        return fb.deemph_fallbacks()


@pytest.mark.parametrize("fma", [False, True])
@pytest.mark.parametrize("name", ["stereo192", "stereo240", "mono192", "drop192", "nolpr192"])
def test_mixed_batch_equals_the_restatement(name, fma):
    """-X, the default 240 kHz with its in-place quirk, -Y (warp-specialised mono kernel), lpr.mode 0, rate_out2 0."""
    run_mixed(CONFIGS[name], P, fma=fma)


def test_explicit_pole_equals_a_handle_created_with_it():
    kw = CONFIGS["stereo192"]
    iq = captures(kw, 3, 2)
    with R.FmBatch(R.DemodConfig(**kw, n_streams=3)) as fb:
        fb.set_stream_output(deemph_lambda=[0.0, 0.9, 0.5], volume=[0.4, 0.7, 0.4])
        lam = fb.stream_output()["lambda"]
        assert lam[1] == np.float32(0.9) and lam[2] == np.float32(0.5) and lam[0] == fb.tables()["misc"][2]
        got = fb.run(iq)
    for s, (lam, vol) in enumerate([(0.0, 0.4), (0.9, 0.7), (0.5, 0.4)]):
        with R.FmBatch(R.DemodConfig(**kw, n_streams=1, deemph_lambda=lam, volume=vol)) as one:
            assert one.deemph_kernel_name() == "fmb_deemph_kernel"
            assert np.array_equal(got[s], one.run(iq[s:s + 1])[0]), f"stream {s}"


@pytest.mark.parametrize("n_streams,seq,shift", [(1, (16, 1, 16), 3), (1, (64,), 2), (1, (16,), 1), (8, (16, 1, 16), 0),
                                                (8, (64,), 5)])
def test_segmented_de_emphasis_per_stream(n_streams, seq, shift):
    """Rows split into time segments: a stream switched off passes its values through, a pole near 1 is repaired."""
    fallbacks = run_mixed(CONFIGS["stereo192"], n_streams, seq=seq, shift=shift)
    if any(setting(s + shift)[0] == 1.0 for s in range(n_streams)):
        assert fallbacks > 0, "the pole near 1 must make the junction walk repair segments"
    elif n_streams == 1 and setting(shift)[0] == 0.0:
        assert fallbacks == 0, "a stream switched off has nothing to repair"


def test_a_pole_near_one_repairs_only_its_own_stream():
    kw = CONFIGS["stereo192"]
    iq = captures(kw, 4, 16)
    counts = []
    for near in (None, 2):
        with R.FmBatch(R.DemodConfig(**kw, n_streams=4, max_blocks_per_call=16)) as fb:
            if near is not None:
                fb.set_stream_output(deemph=1.0, first=near)
                fb.set_stream_output(deemph=[0.000050], first=near + 1)
                assert fb.deemph_kernel_name() == "fmb_deemph_seg_kernel_per_stream"
            pcm = fb.process(np.ascontiguousarray(iq))
            counts.append(fb.deemph_fallbacks())
        for s in range(4):
            want = oracle(kw, 1.0 if s == near else 0.000050, 0.4).run(iq[s])
            assert np.array_equal(pcm[s], want), f"stream {s}"
    assert counts[1] > counts[0]


class Model:
    """One restatement per stream; a change of settings hands the old one's state to a new one."""

    def __init__(self, kw, n):
        self.kw = kw
        self.set = [(kw.get("deemph", 0.000050), kw.get("volume", 0.4))] * n
        self.orcs = [oracle(kw, *s) for s in self.set]

    def change(self, s, deemph=None, volume=None):
        d, v = self.set[s]
        d, v = (d if deemph is None else deemph), (v if volume is None else volume)
        o = oracle(self.kw, d, v)
        o.set_state(*self.orcs[s].state())
        self.orcs[s], self.set[s] = o, (d, v)

    def step(self, iq):
        return [o.block(iq[s]) for s, o in enumerate(self.orcs)]


def test_settings_change_between_calls_reset_and_set_volume():
    kw, n = CONFIGS["stereo192"], 4
    iq = captures(kw, n, 8)
    blk = lambda k: np.ascontiguousarray(iq[:, k * B:(k + 1) * B])
    m = Model(kw, n)
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n)) as fb:
        def step(k, where):
            want = m.step(blk(k))
            got = fb.process(blk(k))
            for s in range(n):
                assert np.array_equal(got[s], want[s]), f"{where}: stream {s}"
        step(0, "uniform")
        fb.set_stream_output(volume=[-1.5, 40.0], deemph=[0.0, 0.000075], first=1)
        m.change(1, 0.0, -1.5)
        m.change(2, 0.000075, 40.0)
        step(1, "after the first change")
        fb.set_stream_output(deemph=1.0, first=3)
        m.change(3, deemph=1.0)
        fb.set_stream_output(deemph=[0.000050], first=1)      # back on: carries on from the memory it left
        m.change(1, deemph=0.000050)
        step(2, "after the second change")
        fb.set_volume(0.25)
        for s in range(n):
            m.change(s, volume=0.25)
        assert np.array_equal(fb.stream_output()["volume"], np.full(n, 0.25, np.float32))
        assert fb.deemph_kernel_name() == "fmb_deemph_kernel_per_stream"
        step(3, "after fmb_set_volume")
        before = fb.stream_output()
        fb.reset()
        after = fb.stream_output()
        assert all(np.array_equal(before[k], after[k]) for k in before), "fmb_reset keeps the settings"
        m = Model(kw, n)
        for s, (d, v) in enumerate([(0.000050, 0.25), (0.000050, 0.25), (0.000075, 0.25), (1.0, 0.25)]):
            m.change(s, d, v)
        step(4, "after fmb_reset")
        fb.set_stream_output(deemph=0.000050, deemph_lambda=0.0)
        fb.set_volume(0.4)
        assert fb.deemph_kernel_name() == "fmb_deemph_kernel", "settings set back: the uniform launch again"
        fb.reset()
        got = fb.run(iq[:, :3 * B])
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n)) as fresh:
        assert np.array_equal(got, fresh.run(iq[:, :3 * B]))


def test_pipelined_submits_keep_the_settings_they_were_submitted_with():
    kw, n, steps = CONFIGS["mono192"], 5, 7
    iq = captures(kw, n, steps)
    m = Model(kw, n)
    changes = {1: (0, 0.0, -1.5), 2: (1, 1.0, 40.0), 3: (4, 0.000075, 0.0), 5: (0, 0.000050, 0.4), 6: (4, 0.0, 0.4)}
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n)) as fb:
        pitch = (fb.max_out + 7) & ~7
        ins = [R.pinned_array((n, B), np.uint8) for _ in range(3)]
        outs = [R.pinned_array((n, pitch), np.int16) for _ in range(3)]
        tickets, wants, counts = {}, {}, {}
        for k in range(steps):
            if k >= 3:
                fb.wait(tickets[k - 3])
                got = outs[(k - 3) % 3]
                for s in range(n):
                    assert np.array_equal(got[s, :counts[k - 3]], wants[k - 3][s]), f"step {k - 3}, stream {s}"
            if k in changes:
                s, d, v = changes[k]
                fb.set_stream_output(volume=[v], deemph=[d], first=s)
                m.change(s, d, v)
            ins[k % 3][...] = iq[:, k * B:(k + 1) * B]
            counts[k] = fb.next_out_count()
            wants[k] = m.step(iq[:, k * B:(k + 1) * B])
            tickets[k] = fb.submit(ins[k % 3].ctypes.data, B, outs[k % 3].ctypes.data, pitch)
        for k in range(steps - 3, steps):
            fb.wait(tickets[k])
            for s in range(n):
                assert np.array_equal(outs[k % 3][s, :counts[k]], wants[k][s]), f"step {k}, stream {s}"
        for a in ins + outs:
            R.free_pinned(a)


def test_device_resident_calls_snapshot_the_settings():
    """fmb_process_device back to back without a host sync, the settings changed before every call."""
    import torch
    kw, n, steps = CONFIGS["stereo192"], 3, 6
    iq = captures(kw, n, steps)
    m = Model(kw, n)
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n)) as fb:
        pitch = (fb.max_out + 7) & ~7
        d_iq = torch.from_numpy(np.ascontiguousarray(iq)).cuda()
        d_pcm = [torch.zeros((n, pitch), dtype=torch.int16, device="cuda") for _ in range(steps)]
        torch.cuda.synchronize()                          # the handle's stream does not wait for torch's
        st = R.lib().fmb_internal_stream(fb._h)
        wants, counts = [], []
        for k in range(steps):
            s, d, v = k % n, DEEMPH[k % 4], VOLUME[(k + 1) % 4]
            fb.set_stream_output(volume=[v], deemph=[d], first=s)
            m.change(s, d, v)
            counts.append(fb.next_out_count())
            wants.append(m.step(iq[:, k * B:(k + 1) * B]))
            fb.process_device(d_iq.data_ptr() + k * B, steps * B, d_pcm[k].data_ptr(), pitch, st)
        L.check(R.lib().fmb_sync(fb._h), "fmb_sync")
        for k in range(steps):
            got = d_pcm[k].cpu().numpy()
            for s in range(n):
                assert np.array_equal(got[s, :counts[k]], wants[k][s]), f"call {k}, stream {s}"


@pytest.mark.parametrize("n_streams,env", [(1, {}), (31, {}), (97, {}), (1024, {}),
                                           (1024, {"FMB_CHUNK": "2", "FMB_TAIL_PCT": "50"}),
                                           (97, {"FMB_PDL": "0"}), (1024, {"FMB_PDL": "0"}), (1024, {"FMB_PDL": "1"})])
def test_work_assignment_regimes(monkeypatch, n_streams, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    run_mixed(CONFIGS["stereo192"], n_streams, seq=(1, 1, 1), shift=1 if n_streams == 1 else 0)


def test_refusals_leave_nothing_half_applied():
    with R.FmBatch(R.DemodConfig(n_streams=4)) as fb:
        before = fb.stream_output()
        bad = [dict(volume=[1.0, np.nan]), dict(volume=[np.inf]), dict(deemph=[0.0001, -1e-6]), dict(deemph=[np.nan]),
               dict(deemph_lambda=[0.5, 1.0]), dict(deemph_lambda=[-0.1]), dict(volume=[1.0] * 3, first=2),
               dict(volume=[1.0], first=4), dict(volume=[1.0], first=-1)]
        for kw in bad:
            with pytest.raises(L.FmbError) as e:
                fb.set_stream_output(**kw)
            assert e.value.code == L.FMB_ERR_ARG, kw
            after = fb.stream_output()
            assert all(np.array_equal(before[k], after[k]) for k in before), kw
        fb.set_stream_output(volume=[-3.0], first=3)        # negative volumes stay allowed, as in fmb_set_volume
        assert fb.stream_output(3, 1)["volume"][0] == -3.0
        assert fb.deemph_kernel_name() == "fmb_deemph_kernel_per_stream"


def test_multi_gpu_host_with_a_range_across_shards():
    kw = CONFIGS["stereo192"]
    n_dev = R.device_count()
    devices = list(range(3)) if n_dev >= 3 else [0, 0, 0]
    n = 13
    iq = captures(kw, n, 2)
    d = [DEEMPH[s % 4] for s in range(2, 11)]
    v = [VOLUME[(s + 1) % 4] for s in range(2, 11)]
    with R.FmMulti(R.DemodConfig(**kw, n_streams=n), devices) as fm:
        assert [c for _, c, _ in fm.shards] == [4, 4, 5]
        with pytest.raises(L.FmbError):
            fm.set_stream_output(volume=[1.0] * 3, first=11)
        with pytest.raises(L.FmbError):
            fm.set_stream_output(volume=[1.0] * 9 + [np.nan], first=2)
        assert np.array_equal(fm.stream_output()["volume"], np.full(n, 0.4, np.float32)), "nothing applied"
        fm.set_stream_output(volume=v, deemph=d, first=2)
        so = fm.stream_output()
        assert np.array_equal(so["volume"][2:11], np.array(v, np.float32))
        assert np.array_equal(so["deemph_on"][2:11], np.array(d) != 0)
        part = fm.stream_output(3, 6)
        assert np.array_equal(part["volume"], so["volume"][3:9])
        stage = R.pinned_array((n, 2 * B), np.uint8)
        stage[...] = iq
        fm.set_blocks_per_call(1)
        got = np.concatenate([fm.process(np.ascontiguousarray(stage[:, k * B:(k + 1) * B])).copy() for k in range(2)],
                             axis=1)
        R.free_pinned(stage)
    for s in range(n):
        ds, vs = (d[s - 2], v[s - 2]) if 2 <= s < 11 else (0.000050, 0.4)
        assert np.array_equal(got[s], oracle(kw, ds, vs).run(iq[s])), f"stream {s}"


def test_player_manifest_matches_single_channel_runs(tmp_path):
    player = os.path.join(ROOT, "rtl_fm_player_b200", "fmb_player")
    kw = CONFIGS["stereo192"]
    chans = [("0.4", "50"), ("1.5", "75"), ("-0.5", "0")]
    files = []
    for i, blocks in enumerate([5, 7, 6]):
        p = tmp_path / f"cap{i}.u8"
        R.synth.capture("fm_stereo", i, kw["rate_in"], 0, blocks * B // 2).tofile(p)
        files.append(str(p))
    single = {}
    for i, (v, e) in enumerate(chans):
        d = tmp_path / f"single{i}"
        d.mkdir()
        r = subprocess.run([player, "-X", "-v", v, "-e", e, "-o", str(d), files[i]], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        single[os.path.basename(files[i]) + ".pcm"] = (d / (os.path.basename(files[i]) + ".pcm")).read_bytes()
    man = tmp_path / "channels.txt"
    man.write_text("# path volume deemph_us\n" + "".join(f"{f} {v} {e}\n" for f, (v, e) in zip(files, chans)))
    for K in (1, 4):
        d = tmp_path / f"manifest_K{K}"
        d.mkdir()
        r = subprocess.run([player, "-X", "-K", str(K), "-o", str(d), "-M", str(man)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        got = {f.name: f.read_bytes() for f in d.iterdir()}
        assert got.keys() == single.keys()
        for k in single:
            assert got[k] == single[k], f"-K {K}: {k}"
    want = oracle(kw, 0.000075, 1.5).run(np.fromfile(files[1], dtype=np.uint8))
    assert single[os.path.basename(files[1]) + ".pcm"] == want.tobytes()


def test_per_stream_passes_write_nothing_outside_the_pcm_rows():
    """Segmented and one-block per-stream passes, settings changed before every device-resident call and the calls
    enqueued back to back: every int16 past a row's out count, in the row padding and in a guard row after the last
    stream keeps its fill pattern, and the rows equal the restatement."""
    import torch
    kw, n, blocks = CONFIGS["stereo192"], 8, 16
    seq = [16, 1, 16, 3]
    iq = captures(kw, n, sum(seq))
    m = Model(kw, n)
    fill = 0x5A5A
    with R.FmBatch(R.DemodConfig(**kw, n_streams=n, max_blocks_per_call=blocks)) as fb:
        pitch = ((fb.max_out + 7) & ~7) + 64
        d_iq = torch.from_numpy(np.ascontiguousarray(iq)).cuda()
        d_pcm = [torch.full((n + 1, pitch), fill, dtype=torch.int16, device="cuda") for _ in seq]
        torch.cuda.synchronize()
        st = R.lib().fmb_internal_stream(fb._h)
        wants, counts, off = [], [], 0
        for k, nb in enumerate(seq):
            for s in range(n):
                d, v = DEEMPH[(s + k) % 4], VOLUME[(s + 2 * k) % 4]
                m.change(s, d, v)
                fb.set_stream_output(volume=[v], deemph=[d], first=s)
            fb.set_blocks_per_call(nb)
            counts.append(fb.next_out_count())
            wants.append([np.concatenate([o.block(iq[s, (off + b) * B:(off + b + 1) * B]) for b in range(nb)])
                          for s, o in enumerate(m.orcs)])
            fb.process_device(d_iq.data_ptr() + off * B, iq.shape[1], d_pcm[k].data_ptr(), pitch, st)
            off += nb
        L.check(R.lib().fmb_sync(fb._h), "fmb_sync")
        assert fb.deemph_fallbacks() > 0
    for k in range(len(seq)):
        got = d_pcm[k].cpu().numpy()
        assert (got[:, counts[k]:].view(np.uint16) == fill).all(), f"call {k}: a write past the out count"
        assert (got[n].view(np.uint16) == fill).all(), f"call {k}: a write into the guard row"
        for s in range(n):
            assert np.array_equal(got[s, :counts[k]], wants[k][s]), f"call {k}, stream {s}"


def test_player_de_emphasis_flag_holds_wherever_the_preset_stands(tmp_path):
    player = os.path.join(ROOT, "rtl_fm_player_b200", "fmb_player")
    kw = CONFIGS["stereo192"]
    cap = tmp_path / "cap.u8"
    R.synth.capture("fm_stereo", 0, kw["rate_in"], 0, 3 * B // 2).tofile(cap)
    outs = []
    for args in (["-e", "0", "-X"], ["-X", "-e", "0"]):
        d = tmp_path / f"out{len(outs)}"
        d.mkdir()
        r = subprocess.run([player] + args + ["-o", str(d), str(cap)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append((d / "cap.u8.pcm").read_bytes())
    assert outs[0] == outs[1] == oracle(kw, 0.0, 0.4).run(np.fromfile(cap, dtype=np.uint8)).tobytes()
