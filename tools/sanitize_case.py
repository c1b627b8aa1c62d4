"""Small end-to-end case for compute-sanitizer (memcheck / racecheck / initcheck / synccheck):
stereo 240 kHz (quirk path, ragged de-emphasis chunks), 5 streams x 3 blocks, plus mono (4:1 and generic tick path of the
warp-specialised kernel) and the drop-sample mode; the dynamic work assignment and overlapping launches; per-stream output
settings on segmented multi-block rows, changed between device-resident calls."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rtl_fm_player_b200 as R
from oracle.oracle_py import PortOracle

B = 262144
for kw, kind in ((dict(rate_in=240000, rate_out2=48000, mode=2, size=90), "random"),
                 (dict(rate_in=192000, rate_out2=48000, mode=1, size=128), "fm_mono"),
                 (dict(rate_in=240000, rate_out2=48000, mode=1, size=128), "fm_mono"),   # warp-specialised kernel, generic tick path
                 (dict(rate_in=192000, rate_out2=48000, mode=0, size=90), "fm_stereo")):
    n, blocks = 5, 3
    iq = np.stack([R.synth.capture(kind, s, kw["rate_in"], 0, blocks * B // 2) for s in range(n)])
    with R.FmBatch(R.DemodConfig(n_streams=n, **kw)) as fb:
        pcm = fb.run(iq)
    for s in range(n):
        assert np.array_equal(pcm[s], PortOracle(**kw).run(iq[s])), (kw, s)
# the dynamic work assignment (a batch that fills the GPU): whole-stream runs chained through shared memory,
# fine-grain runs with lead-ins, the named-barrier hand-overs, on random bytes
os.environ["FMB_CHUNK"], os.environ["FMB_TAIL_PCT"] = "2", "30"
kw = dict(rate_in=192000, rate_out2=48000, mode=2, size=90)
n, uniq = 60, 3
iq = np.stack([R.synth.capture("random", s % uniq, 192000, 0, B // 2) for s in range(n)])
with R.FmBatch(R.DemodConfig(n_streams=n, **kw)) as fb:
    pcm = fb.run(iq)
want = [PortOracle(**kw).run(iq[s]) for s in range(uniq)]
for s in range(n):
    assert np.array_equal(pcm[s], want[s % uniq]), ("dynamic", s)
# round 2: overlapping launches (programmatic dependent launch: per-stream hand-over counters, whole-stream tickets)
# and the warp-specialised mono kernel (producer/consumer named barriers), device-resident back to back
import torch
del os.environ["FMB_CHUNK"], os.environ["FMB_TAIL_PCT"]
for kw, kind, n in ((dict(rate_in=192000, rate_out2=48000, mode=2, size=90), "fm_stereo", 40),
                    (dict(rate_in=192000, rate_out2=48000, mode=1, size=128), "fm_mono", 40),
                    (dict(rate_in=250000, rate_out2=44100, mode=1, size=90), "fm_mono", 40)):
    blocks, uniq = 3, 2
    os.environ["FMB_CHUNK"], os.environ["FMB_TAIL_PCT"] = "8", "0"      # force the ticketed path on a small batch
    iq = np.stack([R.synth.capture(kind, s % uniq, kw["rate_in"], 0, blocks * B // 2) for s in range(n)])
    d_in = torch.from_numpy(iq).cuda()
    with R.FmBatch(R.DemodConfig(n_streams=n, **kw)) as fb:
        n_out = fb.next_out_count()
        pitch = (n_out + 7) & ~7
        d_out = torch.zeros((blocks, n, pitch), dtype=torch.int16, device="cuda")
        st = torch.cuda.Stream()
        for b in range(blocks):
            fb.process_device(d_in.data_ptr() + b * B, iq.shape[1], d_out[b].data_ptr(), pitch, st.cuda_stream)
        fb.join(st.cuda_stream)
        torch.cuda.synchronize()
    got = np.concatenate([d_out[b, :, :n_out].cpu().numpy() for b in range(blocks)], axis=1)
    want = [PortOracle(**kw).run(iq[s]) for s in range(uniq)]
    for s in range(n):
        assert np.array_equal(got[s], want[s % uniq]), ("overlap", kw["mode"], s)
# per-stream output settings: 8 stereo streams x 16 blocks per call (segmented de-emphasis with its junction walk), the
# settings changed between device-resident calls so that each call uploads its own table ahead of its pass: 50 us,
# 75 us, off and a pole near 1 (1 s: the repair path), volumes 0.4, -1.5, 40 and 0
for k in ("FMB_CHUNK", "FMB_TAIL_PCT"):
    os.environ.pop(k, None)
kw = dict(rate_in=192000, rate_out2=48000, mode=2, size=90)
n, blocks, calls = 8, 16, 3
iq = np.stack([R.synth.capture("fm_stereo", s, kw["rate_in"], 0, calls * blocks * B // 2) for s in range(n)])
d_in = torch.from_numpy(iq).cuda()
deemph = [0.000050, 0.000075, 0.0, 1.0]
volume = [0.4, -1.5, 40.0, 0.0]
orcs = [PortOracle(**kw) for _ in range(n)]
with R.FmBatch(R.DemodConfig(n_streams=n, max_blocks_per_call=blocks, **kw)) as fb:
    pitch = (fb.max_out + 7) & ~7
    d_out = torch.zeros((calls, n, pitch), dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    counts, wants = [], []
    for c in range(calls):
        sd = [deemph[(s + c) % 4] for s in range(n)]
        sv = [volume[(s + 2 * c) % 4] for s in range(n)]
        fb.set_stream_output(deemph=sd, volume=sv)
        for s in range(n):                                 # the restatement carries on under the new settings
            o = PortOracle(**kw, deemph=sd[s], volume=sv[s])
            o.set_state(*orcs[s].state())
            orcs[s] = o
        assert fb.deemph_kernel_name() == "fmb_deemph_seg_kernel_per_stream"
        counts.append(fb.next_out_count())
        fb.process_device(d_in.data_ptr() + c * blocks * B, iq.shape[1], d_out[c].data_ptr(), pitch, st.cuda_stream)
        wants.append([orcs[s].run(iq[s, c * blocks * B:(c + 1) * blocks * B]) for s in range(n)])
    fb.join(st.cuda_stream)                                # the calls ran back to back, each with its own table
    torch.cuda.synchronize()
    for c in range(calls):
        got = d_out[c, :, :counts[c]].cpu().numpy()
        for s in range(n):
            assert np.array_equal(got[s], wants[c][s]), ("per-stream output", c, s)
    assert fb.deemph_fallbacks() > 0
print("sanitize case ok")
