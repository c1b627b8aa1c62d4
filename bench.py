#!/usr/bin/env python
"""bench.py -- throughput of the batched IQ -> PCM path (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, libfmb.so)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU code, all host cores

A step = one pass of the hot path over one batch: every stream of the rank's shard consumes one
reference block (262144 bytes = 131072 IQ samples, rtl_fm_player.h:31-33) and produces its PCM.
Headline workload = BASELINE.json configs[3]: 1024 stereo FM streams per GPU, -X preset (192 kHz -> 48 kHz
stereo, 90 taps), rotate path ("scaling": "weak").  The same run also times configs[4] as stated -- 8192
streams in total, sharded 8192/N per GPU ("strong" object; `--scaling strong` makes it the headline) --
checks 8 streams of every rank's shard against the CPU oracle outside the timed regions ("parity"), reports a
roofline entry per kernel from separate profiling passes, and measures end to end through the C multi-GPU host
(fmb_multi: one process, one worker thread per device, one pinned buffer) next to the box's raw copy ceiling.
Prints ONE JSON line on rank 0.

    python bench.py --gpus 1 --steps K --warmup W --dump-outputs bench_outputs

also writes the PCM of the headline's last timed step, as float32 .npy files (see dump_outputs), so that two
builds run with the same arguments -- hence the same synthetic inputs -- can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK = 262144                    # bytes per stream per step (MAXIMUM_BUF_LENGTH)
SAMPLES_PER_BLOCK = BLOCK // 2
ALG_BYTES = {"stereo": 2.125, "mono": 2.0625}   # SURVEY.md s8(d): u8 IQ in + int16 PCM out per IQ sample
# the de-emphasis kernel's own compulsory traffic: f32 decoder output in (L,R at 48 kHz: 8 B per 32 IQ samples; mono 4 B),
# int16 PCM out (4 B resp. 2 B per 32 IQ samples)
DEEMPH_ALG_BYTES = {"stereo": 0.375, "mono": 0.1875}
FP32_OPS_PER_SAMPLE = {"stereo": 69.0, "mono": 23.0}  # bit-exact (no FMA) FP32 instructions per IQ sample, SURVEY s8(d)
METRIC = "aggregate IQ Msamples/s to stereo PCM"
UNIT = "Msamples/s"


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, streams, mode, precision):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this
    kernel (profiles/kernel_traffic.json names the .ncu-rep summary it was read from).  ncu cannot run inside a
    benchmark, so this is the one number of the line that is not measured live; it is only attached to the
    workload it was captured on, null otherwise."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernel_traffic.json")) as f:
            t = json.load(f)[kernel]
        if streams == t["streams"] and mode == t["mode"] and precision == t["precision"]:
            return t["traffic"], t["source"]
    except Exception:
        pass
    return None, None


def load_synth():
    """rtl_fm_player_b200/synth.py loaded as a stand-alone module: it maps only libfmsynth.so (plain C), so the
    reference arm generates its captures without importing the package or mapping the product library."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("fm_synth_only", os.path.join(ROOT, "rtl_fm_player_b200", "synth.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, sampled through NVML every ~0.5 ms
    (nvidia-smi, one process per sample, is too slow for a region of a few milliseconds; it is the
    fallback)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.samples, self._stop, self._t = index, [], threading.Event(), None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES if it is a plain list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                phys = int(vis.split(",")[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.bits = [(pynvml.nvmlClocksEventReasonHwSlowdown if hasattr(pynvml, "nvmlClocksEventReasonHwSlowdown") else 0x8),
                         0x40, 0x20, 0x4]  # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        except Exception:
            self.nvml = None

    def _run(self):
        while not self._stop.is_set():
            try:
                if self.nvml is not None:
                    mhz = float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
                    try:
                        mask = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        mask = int(self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    self.samples.append([str(mhz), str(self.max_mhz)] + ["Active" if mask & b else "Not Active" for b in self.bits])
                    self._stop.wait(0.0005)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = sorted({n for s in self.samples for n, v in zip(self.NAMES, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own rtl_fm_player.c (oracle/_ref/ref_offline)
# ------------------------------------------------------------------------------------------
def cpu_reference_run(mode: str, target_seconds: float, cores: int | None = None):
    """One reference process per core, each demodulating its own preloaded capture
    (BASELINE.md s3).  Returns dict(value Msamples/s, cores, kind, sample, seconds)."""
    synth = load_synth()
    cli = os.path.join(ROOT, "oracle", "_ref", "ref_offline")
    kind = "reference"
    if not os.path.exists(cli):
        return cpu_port_run(mode, target_seconds, cores)
    cores = cores or os.cpu_count() or 1
    flag = "-X" if mode == "stereo" else "-Y"
    nblk = 4
    tmp = tempfile.mkdtemp(prefix="fmref_")
    files = []
    for c in range(min(cores, 8)):  # 8 distinct captures, reused round-robin
        fn = os.path.join(tmp, f"s{c}.u8")
        synth.capture("fm_stereo" if mode == "stereo" else "fm_mono", c, 192000, 0, nblk * SAMPLES_PER_BLOCK).tofile(fn)
        files.append(fn)
    # calibrate one process
    t0 = time.perf_counter()
    subprocess.run([cli, flag, "-n", "8", files[0]], capture_output=True, text=True, check=True)
    per_rep = (time.perf_counter() - t0) / 8
    reps = max(4, int(target_seconds / max(per_rep, 1e-4)))
    t0 = time.perf_counter()
    procs = [subprocess.Popen([cli, flag, "-n", str(reps), files[c % len(files)]], stdout=subprocess.PIPE, text=True)
             for c in range(cores)]
    outs = [p.communicate()[0] for p in procs]
    wall = time.perf_counter() - t0
    samples, dsp_max = 0, 0.0
    for o in outs:
        for tok in o.split():
            if tok.startswith("samples="):
                samples += int(tok[8:])
            if tok.startswith("dsp_s="):
                dsp_max = max(dsp_max, float(tok[6:]))
    for fn in files:
        os.unlink(fn)
    os.rmdir(tmp)
    return {"value": samples / wall * 1e-6, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{cores} reference processes (oracle/_ref/ref_offline {flag}), each {reps}x a {nblk}-block synthetic capture "
                      f"({reps * nblk} blocks of 131072 IQ samples), whole-process wall {wall:.1f}s, slowest DSP-only {dsp_max:.1f}s",
            "seconds": wall, "dsp_only_value": samples / max(dsp_max, 1e-9) * 1e-6}


def cpu_port_run(mode: str, target_seconds: float, cores: int | None = None):
    """Fallback when oracle/_ref was not built: the C restatement, one thread per core."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle.oracle_py import PortOracle
    synth = load_synth()
    cores = cores or os.cpu_count() or 1
    kw = dict(rate_in=192000, rate_out2=48000, mode=2 if mode == "stereo" else 1, size=90 if mode == "stereo" else 128)
    iq = synth.capture("fm_stereo" if mode == "stereo" else "fm_mono", 0, 192000, 0, 4 * SAMPLES_PER_BLOCK)
    o = PortOracle(**kw)
    t0 = time.perf_counter(); o.bench(iq, 2); per_rep = (time.perf_counter() - t0) / 2
    reps = max(2, int(target_seconds / per_rep))
    orcs = [PortOracle(**kw) for _ in range(cores)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=cores) as ex:   # ctypes releases the GIL
        samples = sum(ex.map(lambda oo: oo.bench(iq, reps), orcs))
    wall = time.perf_counter() - t0
    return {"value": samples / wall * 1e-6, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{cores} threads of oracle/fm_oracle.c, each {reps}x a 4-block capture, wall {wall:.1f}s", "seconds": wall}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps, warm = max(1, args.steps), max(0, args.warmup)
    per_step = max(1.0, min(8.0, 60.0 / (steps + warm)))
    for _ in range(warm):
        cpu_reference_run(args.mode, per_step)
    vals, last = [], None
    t0 = time.perf_counter()
    for _ in range(steps):
        last = cpu_reference_run(args.mode, per_step)
        vals.append(last["value"])
    wall = time.perf_counter() - t0
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": wall / steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "maps_product_library": "libfmb.so" in open("/proc/self/maps").read(),
    }
    emit(line)
    return 0


def headline_streams(args, world):
    """streams per GPU of the headline measurement"""
    return args.streams if args.scaling == "weak" else max(1, args.total_streams // world)


def workload_config(args, world):
    S = headline_streams(args, world)
    cfg = "configs[3] (1024 streams per GPU)" if args.scaling == "weak" else f"configs[4] ({args.total_streams} streams sharded over {world} GPU(s))"
    return {"workload": f"{S} {args.mode} FM streams per GPU x 1 reference block (262144 B = 131072 IQ samples) per step; "
                        f"{'-X' if args.mode == 'stereo' else '-Y'} preset (192 kHz -> 48 kHz, "
                        f"{'90-tap stereo' if args.mode == 'stereo' else '128-tap mono'}), rotate_90 path; BASELINE.json {cfg}",
            "streams_per_gpu": S, "block_bytes": BLOCK, "precision": args.precision, "segments": args.segments,
            "l2": f"{args.nbuf} distinct {S * BLOCK >> 20} MiB input batches in rotation (each > 126 MB L2), no flush needed"}


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import rtl_fm_player_b200 as R

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    numa_node = R.lib().fmb_bind_thread_to_device_node(local)   # pinned buffers below become node-local
    dist, host_group = None, None
    if world > 1:
        import torch.distributed as dist
        backend = os.environ.get("FMB_BENCH_BACKEND", "nccl")
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
        host_group = dist.new_group(backend="gloo")       # host-side barriers/gathers that must not touch the GPUs
    red_dev = "cuda" if dist is None or dist.get_backend() == "nccl" else "cpu"

    K, W = args.steps, max(3, args.warmup)
    stereo = args.mode == "stereo"
    mk = R.DemodConfig.stereo_192k if stereo else R.DemodConfig.mono_192k
    okw = dict(rate_in=192000, rate_out2=48000, mode=2 if stereo else 1, size=90 if stereo else 128)
    prec = R.FMB_PRECISION_FMA if args.precision == "fma" else R.FMB_PRECISION_EXACT
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return float(x)
        t = torch.tensor([float(x)], device=red_dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- synthetic input: `uniq` distinct channels per rank (global stream ids), nbuf consecutive blocks of each;
    # a shard of S streams holds them round-robin (stream s carries channel s % uniq), replicated ON the device ----
    S_weak = args.streams
    S_strong = max(1, args.total_streams // world)
    S_head = headline_streams(args, world)
    uniq = min(args.unique, S_weak, S_strong)
    kind = "fm_stereo" if stereo else "fm_mono"
    host_uniq = np.empty((args.nbuf, uniq, BLOCK), dtype=np.uint8)
    def gen(u, base):
        cap = R.synth.capture(kind, base + u, 192000, 0, args.nbuf * SAMPLES_PER_BLOCK)
        for b in range(args.nbuf):
            host_uniq[b, u] = cap[b * BLOCK:(b + 1) * BLOCK]
    from concurrent.futures import ThreadPoolExecutor
    data_rank = int(os.environ.get("FMB_BENCH_DATA_RANK", rank))     # (override: time another rank's channels on one GPU)
    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        list(ex.map(lambda u: gen(u, data_rank * args.unique), range(uniq)))
    dev_uniq = torch.from_numpy(host_uniq).cuda()

    def device_inputs(S):
        idx = torch.arange(S, device="cuda") % uniq
        return [dev_uniq[b].index_select(0, idx).contiguous() for b in range(args.nbuf)]

    def time_resident(S, precision):
        """K timed steps of S streams per GPU, inputs resident in HBM; returns (ms over the K steps as max over
        ranks, host enqueue seconds, launches, clocks, PCM count per stream of the last step)."""
        fb = R.FmBatch(mk(n_streams=S, device=local, precision=precision, segments=args.segments))
        n_out = fb.next_out_count()
        pitch = (n_out + 7) & ~7
        dev_in = device_inputs(S)
        dev_pcm = torch.empty((S, pitch), dtype=torch.int16, device="cuda")
        for i in range(W):
            fb.process_device(dev_in[i % args.nbuf].data_ptr(), BLOCK, dev_pcm.data_ptr(), pitch, stream)
        fb.join(stream)
        barrier()
        launches0 = R.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clk:
            barrier()
            e0.record()
            t_host = time.perf_counter()
            for i in range(K):
                if i == K - 1:
                    n_last = fb.next_out_count()           # PCM per stream of the last step (host arithmetic)
                fb.process_device(dev_in[(W + i) % args.nbuf].data_ptr(), BLOCK, dev_pcm.data_ptr(), pitch, stream)
            t_host = time.perf_counter() - t_host       # host time to enqueue the K steps (must stay below the device time)
            fb.join(stream)
            e1.record()
            barrier()
        ms = max_over_ranks(e0.elapsed_time(e1))
        launches = R.launch_count() - launches0
        return fb, dev_in, dev_pcm, pitch, n_out, ms, t_host, launches, clk.summary(), n_last

    # ---- headline: device-resident `value` ----
    fb, dev_in, dev_pcm, pitch, n_out, ms_total, t_host, launches, clocks, n_last = time_resident(S_head, prec)
    value = S_head * world * SAMPLES_PER_BLOCK * K / (ms_total * 1e-3) * 1e-6
    last_pcm = dev_pcm[:, :n_last].cpu().numpy() if args.dump_outputs else None   # the passes below overwrite dev_pcm

    # ---- per-kernel device times, in SEPARATE passes over the same steps (nothing below touches the headline):
    #   pass A: K pipelined steps with an event pair around every demod launch (its steady-state duration)
    #   pass B: K steps with a device synchronisation after each, so that the de-emphasis kernel (side stream,
    #           normally overlapped with the next demod launch and waiting for its SM slots) runs ALONE ----
    demod_kernel = fb.kernel_name()
    # pass A0: K pipelined steps, ONE event pair on the launching stream around the K demod launches (no per-launch
    # events: timing events between the launches perturb their overlap) -> the launch period of the steady state
    for i in range(W):
        fb.process_device(dev_in[i % args.nbuf].data_ptr(), BLOCK, dev_pcm.data_ptr(), pitch, stream)
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(K):
        fb.process_device(dev_in[(W + i) % args.nbuf].data_ptr(), BLOCK, dev_pcm.data_ptr(), pitch, stream)
    p1.record()                                         # behind the last demod launch, before the join
    fb.join(stream)
    torch.cuda.synchronize()
    demod_period_ms = p0.elapsed_time(p1) / K
    fb.profile_enable(True)
    fb.profile_reset()
    for i in range(K):
        fb.process_device(dev_in[i % args.nbuf].data_ptr(), BLOCK, dev_pcm.data_ptr(), pitch, stream)
    fb.join(stream)
    torch.cuda.synchronize()
    prof_a = fb.profile_read()
    fb.profile_reset()
    for i in range(K):
        fb.process_device(dev_in[i % args.nbuf].data_ptr(), BLOCK, dev_pcm.data_ptr(), pitch, stream)
        fb.join(stream)
        torch.cuda.synchronize()
    prof_b = fb.profile_read()
    fb.profile_enable(False)
    # pipelined, consecutive launches overlap (programmatic dependent launch): the event pair around a launch spans
    # from the END of the previous launch to the end of this one, i.e. it is the launch PERIOD of the steady state
    demod_pairs_ms = prof_a["demod_ms"] / max(prof_a["demod_launches"], 1)
    demod_ms = demod_period_ms
    demod_alone_ms = prof_b["demod_ms"] / max(prof_b["demod_launches"], 1)
    deemph_ms = prof_b["deemph_ms"] / max(prof_b["deemph_launches"], 1)

    # ---- parity of THIS rank's shard on THIS GPU, outside every timed region: a fresh handle of the same shard size
    # (same kernels, same work assignment) demodulates the nbuf consecutive blocks; 8 streams spread over the shard
    # -- first and last included -- are compared bit for bit with the CPU oracle (checker only) ----
    def shard_parity(S):
        from oracle.oracle_py import PortOracle
        pf = R.FmBatch(mk(n_streams=S, device=local, precision=prec, segments=args.segments))
        p_in = device_inputs(S) if S != S_head else dev_in
        outs = []
        for b in range(args.nbuf):
            o = torch.empty((S, pitch), dtype=torch.int16, device="cuda")
            pf.process_device(p_in[b].data_ptr(), BLOCK, o.data_ptr(), pitch, stream)
            outs.append(o)
        pf.join(stream)
        torch.cuda.synchronize()
        pick = sorted(set(int(x) for x in np.linspace(0, S - 1, min(8, S))))
        got = np.concatenate([o[pick, :n_out].cpu().numpy() for o in outs], axis=1)
        bad = 0
        for row, s in enumerate(pick):
            want = PortOracle(**okw).run(np.concatenate([host_uniq[b, s % uniq] for b in range(args.nbuf)]))
            if args.precision == "exact":
                bad += int(not np.array_equal(got[row], want))
            else:
                bad += int(np.abs(got[row].astype(np.int32) - want.astype(np.int32)).max() > 1)
        pf.close()
        return bad == 0, len(pick)
    parity_ok, parity_n = shard_parity(S_head)

    # ---- the other scaling mode, same run: configs[4] as stated (total_streams sharded over the GPUs) when the
    # headline is weak, and vice versa ----
    S_other = S_strong if args.scaling == "weak" else S_weak
    other = None
    if not args.no_other_scaling:
        if S_other == S_head:
            other = {"streams_per_gpu": S_other, "value": value, "ms_per_step": ms_total / K, "parity": parity_ok,
                     "note": "same shard size as the headline at this GPU count: one measurement"}
        else:
            fb_o, _, _, _, _, ms_o, _, _, _, _ = time_resident(S_other, prec)
            fb_o.close()
            ok_o, _ = shard_parity(S_other)
            other = {"streams_per_gpu": S_other, "value": S_other * world * SAMPLES_PER_BLOCK * K / (ms_o * 1e-3) * 1e-6,
                     "ms_per_step": ms_o / K, "parity": ok_o}
        other["unit"] = UNIT
        other["total_streams"] = S_other * world

    # ---- the same steps in FMB_PRECISION_FMA (FIR multiply-adds fused: within +-1 LSB of int16 PCM, the
    # tolerance north_star states for the floating-point stages); reported beside the bit-exact headline ----
    fma_alt = None
    if args.precision == "exact" and not args.no_fma_alt:
        fb2, _, _, _, _, fma_ms, _, _, _, _ = time_resident(S_head, R.FMB_PRECISION_FMA)
        fb2.close()
        fma_alt = {"value": S_head * world * SAMPLES_PER_BLOCK * K / (fma_ms * 1e-3) * 1e-6, "unit": UNIT, "ms_per_step": fma_ms / K,
                   "tolerance": "+-1 LSB int16 PCM vs the reference (tests/test_gpu_parity.py::test_fma_precision_within_one_lsb)"}

    # gather the per-rank parity flags on the host side
    parity_flags = [bool(parity_ok)]
    if dist is not None:
        flags = [None] * world
        dist.all_gather_object(flags, bool(parity_ok), group=host_group)
        parity_flags = [bool(f) for f in flags]

    # ---- end to end, per-process layout (round 1's): every rank streams its own shard through fmb_submit/fmb_wait
    # from its own pinned buffers ----
    def e2e_per_process():
        nh = 3
        h_in = [R.pinned_array((S_head, BLOCK), np.uint8, write_combined=True) for _ in range(nh)]
        idx = np.arange(S_head) % uniq
        for b in range(nh):
            h_in[b][...] = host_uniq[b % args.nbuf][idx]
        h_pcm = [R.pinned_array((S_head, pitch), np.int16) for _ in range(R._lib.FMB_PIPE_DEPTH)]
        def loop(n):
            tickets = []
            for i in range(n):
                if len(tickets) >= R._lib.FMB_PIPE_DEPTH:
                    fb.wait(tickets.pop(0))
                tickets.append(fb.submit(h_in[i % nh].ctypes.data, BLOCK, h_pcm[i % len(h_pcm)].ctypes.data, pitch))
            for t in tickets:
                fb.wait(t)
        torch.cuda.synchronize()
        loop(max(3, W))
        barrier()
        t0 = time.perf_counter()
        loop(K)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        for a in h_in + h_pcm:
            R.free_pinned(a)
        return {"value": S_head * world * SAMPLES_PER_BLOCK * K / dt * 1e-6, "unit": UNIT, "ms_per_step": dt / K * 1e3,
                "api": f"{world} process(es), each fmb_submit/fmb_wait on its own shard and pinned buffers, 3 steps in flight"}
    e2e_pp = e2e_per_process() if (world > 1 and not args.no_e2e_per_process) else None

    # ---- everything device-resident is measured: release this rank's GPU memory, then rank 0 alone drives ALL GPUs
    # through the C multi-GPU host (the other ranks wait on the host-side group and leave their GPUs idle) ----
    fb.close()
    del dev_in, dev_pcm, dev_uniq, fb
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier(group=host_group)
    e2e, ceiling = None, None
    if rank == 0:
        from oracle.oracle_py import PortOracle
        n_all = S_head * world
        # all ranks' channels: rank r's shard carries channels r*args.unique + (s % uniq); regenerate the other ranks' here
        host_all = np.empty((args.nbuf, world, uniq, BLOCK), dtype=np.uint8)
        host_all[:, 0] = host_uniq if data_rank == 0 else 0
        def gen_all(ru):
            r, u = divmod(ru, uniq)
            cap = R.synth.capture(kind, r * args.unique + u, 192000, 0, args.nbuf * SAMPLES_PER_BLOCK)
            for b in range(args.nbuf):
                host_all[b, r, u] = cap[b * BLOCK:(b + 1) * BLOCK]
        with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
            list(ex.map(gen_all, range(0 if data_rank else uniq, world * uniq)))
        nh = 3
        with R.FmMulti(mk(n_streams=n_all, precision=prec, segments=args.segments), list(range(world))) as fm:
            h_in = [R.pinned_array((n_all, BLOCK), np.uint8, write_combined=True) for _ in range(nh)]
            h_pcm = [R.pinned_array((n_all, pitch), np.int16) for _ in range(R._lib.FMB_PIPE_DEPTH)]
            idx = np.arange(S_head) % uniq
            for b in range(nh):
                for r in range(world):
                    h_in[b][r * S_head:(r + 1) * S_head] = host_all[b % args.nbuf, r][idx]
            def loop(n):
                tickets = []
                for i in range(n):
                    if len(tickets) >= R._lib.FMB_PIPE_DEPTH:
                        fm.wait(tickets.pop(0))
                    tickets.append(fm.submit(h_in[i % nh].ctypes.data, BLOCK, h_pcm[i % len(h_pcm)].ctypes.data, pitch))
                for t in tickets:
                    fm.wait(t)
            loop(max(3, W))
            fm.sync()
            t0 = time.perf_counter()
            loop(K)
            fm.sync()
            e2e_s = time.perf_counter() - t0
            # parity of the gathered PCM, outside the timed region: restart the streams, demodulate the nh consecutive
            # blocks through the same host path, compare 8 streams of EVERY shard with the oracle
            fm.reset()
            got = []
            for b in range(nh):
                fm.wait(fm.submit(h_in[b].ctypes.data, BLOCK, h_pcm[0].ctypes.data, pitch))
                got.append(h_pcm[0][:, :n_out].copy())
            got = np.concatenate(got, axis=1)
            shard_ok = []
            for r in range(world):
                ok = True
                for s in sorted(set(int(x) for x in np.linspace(0, S_head - 1, min(8, S_head)))):
                    want = PortOracle(**okw).run(np.concatenate([host_all[b, r, s % uniq] for b in range(nh)]))
                    g = got[r * S_head + s]
                    ok &= bool(np.array_equal(g, want)) if args.precision == "exact" else \
                        bool(np.abs(g.astype(np.int32) - want.astype(np.int32)).max() <= 1)
                shard_ok.append(ok)
            checksum = int(got.astype(np.int64).sum())
            for a in h_in + h_pcm:
                R.free_pinned(a)
        h2d, d2h = n_all * BLOCK, n_all * n_out * 2
        e2e = {"value": n_all * SAMPLES_PER_BLOCK * K / e2e_s * 1e-6, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s / K * 1e3,
               "api": f"fmb_multi_submit/fmb_multi_wait (C host, 1 process, {world} worker thread(s), one per GPU), ONE pinned IQ buffer "
                      f"(write-combined) and ONE pinned PCM buffer per step for all GPUs, 3 steps in flight",
               "gbs_h2d": h2d * K / e2e_s * 1e-9, "parity_per_shard": shard_ok, "pcm_checksum": checksum,
               "host_numa_node": numa_node}
        if e2e_pp is not None:
            e2e["per_process_layout"] = e2e_pp
        # raw copy ceiling of the box for the same byte mix, nothing else running (tools/fm_copyprobe.cu)
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import h2d_ceiling
            a, b_, _ = h2d_ceiling.probe(list(range(world)), S_head * BLOCK, max(4, min(K, 10)), 2, 1)
            ceiling = {"gbs_h2d": a, "gbs_d2h": b_, "what": f"{world} concurrent cudaMemcpyAsync streams of {S_head * BLOCK >> 20} MiB "
                       "write-combined pinned H2D + 1/16 of that D2H, no kernels (tools/fm_copyprobe.cu)"}
            e2e["copy_ceiling"] = ceiling
            e2e["copy_ceiling_frac"] = e2e["gbs_h2d"] / a if a > 0 else None
        except Exception as ex_:                              # noqa: BLE001
            e2e["copy_ceiling"] = {"error": str(ex_)}
            e2e["copy_ceiling_frac"] = None

    if last_pcm is not None:                              # every rank writes its own shard
        dump_outputs(args.dump_outputs, last_pcm, "pcm" if world == 1 else f"pcm_rank{rank}", DUMP_BYTES // world)
    if rank != 0:
        if dist is not None:
            dist.barrier(group=host_group)
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak_gbs()
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    fp32_peak = 148 * 128 * sm_mhz * 1e6                         # FP32 lane-instructions/s at the clock seen under load
    samples_launch = S_head * SAMPLES_PER_BLOCK
    def roof(kernel, ms, alg_per_sample, extra=None):
        alg = alg_per_sample * samples_launch
        ach = alg / (ms * 1e-3) * 1e-9
        traffic, src = ncu_traffic(kernel, S_head, args.mode, args.precision)
        d = {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
             "traffic": traffic, "traffic_source": src, "alg_bytes_per_launch": alg, "alg_bytes_per_iq_sample": alg_per_sample,
             "kernel_ms": ms, "peak_source": peak_src}
        if extra:
            d.update(extra)
        return d
    fp32_ach = FP32_OPS_PER_SAMPLE[args.mode] * samples_launch / (demod_ms * 1e-3)
    r_demod = roof(demod_kernel, demod_ms, ALG_BYTES[args.mode], {
        "timing": "kernel_ms = launch period of the steady state: one CUDA-event pair on the launching stream around K back-to-back "
                  "launches (consecutive launches overlap at their ends: programmatic dependent launch), separate pass from the "
                  "headline; kernel_ms_event_pairs = an event pair around every launch (the timing events between the launches "
                  "disturb the overlap); kernel_ms_alone = every launch followed by a device synchronisation",
        "kernel_ms_event_pairs": demod_pairs_ms,
        "kernel_ms_alone": demod_alone_ms,
        "fp32_pipe": {"ops_per_iq_sample": FP32_OPS_PER_SAMPLE[args.mode], "achieved_Tops": fp32_ach * 1e-12,
                      "peak_Tops": fp32_peak * 1e-12, "frac": fp32_ach / fp32_peak,
                      "note": "the path is FP32-issue bound (SURVEY s8d); peak = 148 SM x 128 lanes x SM clock under load"}})
    r_deemph = roof("fmb_deemph_kernel", deemph_ms, DEEMPH_ALG_BYTES[args.mode], {
        "timing": "CUDA events on its own stream with a device synchronisation after every step: the kernel runs alone "
                  "(pipelined it overlaps the next demod launch)",
        "note": "latency-bound recurrence (3 dependent FP32 ops per value), not HBM-bound: its input is the demod kernel's "
                "output, still in L2"})
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": launches, "host_enqueue_ms_per_step": t_host / K * 1e3,
        "parity": {"per_rank": parity_flags, "all": all(parity_flags), "streams_checked_per_rank": parity_n, "blocks": args.nbuf,
                   "against": "oracle/fm_oracle.c (pinned to the reference build), " +
                              ("bit-exact int16 PCM" if args.precision == "exact" else "+-1 LSB int16 PCM"),
                   "where": "each rank's own shard on its own GPU, fresh handle of the same shard size, outside the timed regions"},
        "roofline": r_demod,
        "roofline_kernels": [r_demod, r_deemph],
        ("strong" if args.scaling == "weak" else "weak"): other,
    }
    if fma_alt is not None:
        line["precision_fma"] = fma_alt
    if world == 1 and not args.no_cpu:
        cb = cpu_reference_run(args.mode, args.cpu_seconds)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    else:
        line["cpu_baseline"] = None
    emit(line)
    if dist is not None:
        dist.barrier(group=host_group)
        dist.destroy_process_group()
    return 0


DUMP_BYTES = 64_000_000           # --dump-outputs: at most this much in all


def dump_outputs(out_dir: str, pcm: np.ndarray, name: str, budget: int) -> None:
    """PCM [streams, samples] of one step -> out_dir/<name>.npy (float32, exact for int16) and
    out_dir/<name>_streams.npy (float64 stream indices of its rows).  A batch that would take more than `budget`
    bytes is cut to a fixed, seeded sample of whole streams."""
    S, n = pcm.shape
    keep = max(1, (budget - 256) // (n * 4 + 8))          # a float32 row + its float64 index; 256 B for two headers
    rows = np.arange(S) if keep >= S else np.sort(np.random.default_rng(0).choice(S, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{name}.npy"), pcm[rows].astype(np.float32))
    np.save(os.path.join(out_dir, f"{name}_streams.npy"), rows.astype(np.float64))


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else any library prints (NCCL's version
    banner, ...) was redirected to stderr at start-up."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                     # C-level and Python-level stdout -> stderr from here on
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="headline: weak = --streams per GPU (configs[3]); strong = --total-streams sharded over the GPUs (configs[4])")
    ap.add_argument("--streams", type=int, default=1024, help="streams per GPU (weak scaling)")
    ap.add_argument("--total-streams", type=int, default=8192, help="streams over all GPUs (strong scaling)")
    ap.add_argument("--mode", default="stereo", choices=["stereo", "mono"])
    ap.add_argument("--precision", default="exact", choices=["exact", "fma"])
    ap.add_argument("--segments", type=int, default=0)
    ap.add_argument("--unique", type=int, default=64, help="distinct synthetic channels per GPU (rest are copies)")
    ap.add_argument("--nbuf", type=int, default=4, help="distinct input batches rotated through (each > L2)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-fma-alt", action="store_true", help="skip the extra FMB_PRECISION_FMA timing")
    ap.add_argument("--no-other-scaling", action="store_true", help="skip the second (strong resp. weak) measurement")
    ap.add_argument("--no-e2e-per-process", action="store_true", help="skip the per-process end-to-end layout at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the PCM of the headline's last timed step to DIR/*.npy (float32, at most 64 MiB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
