"""Several blocks per call: what a call of n consecutive blocks per stream buys at few streams, and what it costs at many.

For stereo (-X) and mono (-Y), 1, 8 and 64 streams, at n = 1 and at an n that gives the demod kernel enough work units
to fill the GPU:
  * device-resident rate: IQ already in HBM, fmb_process_device back to back on the handle's stream, host clock around
    a device synchronisation;
  * end-to-end rate: fmb_submit / fmb_wait from pinned host memory with FMB_PIPE_DEPTH calls in flight;
  * kernel 1 and kernel 2 (de-emphasis, the segmented kernel when the row is split into time segments) times per call from the
    handle's own CUDA-event profile, in a separate pass.
Then the work-assignment rule for n > 1 (tickets of one block each versus the static split, forced with FMB_CHUNK /
FMB_TAIL_PCT), and the bench.py headlines (1 024 streams, one block per call) of the parent build and of this one,
alternated in one run.  The card's name and power limit are read in the same run.

usage: python tools/runs_bench.py --out results.json [--parent libfmb_parent.so] [--parent-tree DIR]
--parent-tree is a checkout of the parent commit with its libraries built; without it the A/B is skipped."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rtl_fm_player_b200 import _lib as L  # noqa: E402  (after the path is set)

B = 262144
FILL = {1: 64, 8: 16, 64: 4}          # blocks per call that give >= 2 x 444 work units of 2048 samples


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def make_cfg(R, mode, S, n):
    f = R.DemodConfig.stereo_192k if mode == "stereo" else R.DemodConfig.mono_192k
    return f(n_streams=S, max_blocks_per_call=n)


def inputs(R, mode, S, n, n_bufs):
    kind = "fm_stereo" if mode == "stereo" else "fm_mono"
    u = min(S, 8)
    iq = np.stack([R.synth.capture(kind, s, 192000, 0, n_bufs * n * B // 2) for s in range(u)])
    return iq[np.arange(S) % u]


def device_rate(R, mode, S, n, steps):
    import torch
    n_bufs = 2
    iq = inputs(R, mode, S, n, n_bufs)
    with R.FmBatch(make_cfg(R, mode, S, n)) as fb:
        pitch = (fb.max_out + 7) & ~7
        d_iq = [torch.from_numpy(np.ascontiguousarray(iq[:, k * n * B:(k + 1) * n * B])).cuda() for k in range(n_bufs)]
        d_pcm = torch.empty((S, pitch), dtype=torch.int16, device="cuda")
        st = R.lib().fmb_internal_stream(fb._h)
        for k in range(3):
            fb.process_device(d_iq[k % n_bufs].data_ptr(), n * B, d_pcm.data_ptr(), pitch, st)
        L.check(R.lib().fmb_sync(fb._h), "fmb_sync")
        t0 = time.perf_counter()
        for k in range(steps):
            fb.process_device(d_iq[k % n_bufs].data_ptr(), n * B, d_pcm.data_ptr(), pitch, st)
        L.check(R.lib().fmb_sync(fb._h), "fmb_sync")
        dt = time.perf_counter() - t0
        # kernel times in a pass of their own (event pairs slow the enqueue)
        fb.profile_enable(True)
        fb.profile_reset()
        for k in range(steps):
            fb.process_device(d_iq[k % n_bufs].data_ptr(), n * B, d_pcm.data_ptr(), pitch, st)
        L.check(R.lib().fmb_sync(fb._h), "fmb_sync")
        prof = fb.profile_read()
        kname = fb.kernel_name()
    samples = S * n * (B // 2) * steps
    return {"ms_per_call": dt / steps * 1e3, "Gsamples_per_s": samples / dt * 1e-9,
            "kernel1_ms": prof["demod_ms"] / max(1, prof["demod_launches"]),
            "kernel2_ms": prof["deemph_ms"] / max(1, prof["deemph_launches"]), "kernel": kname}


def e2e_rate(R, mode, S, n, steps):
    iq = inputs(R, mode, S, n, 1)
    with R.FmBatch(make_cfg(R, mode, S, n)) as fb:
        pitch = (fb.max_out + 7) & ~7
        depth = L.FMB_PIPE_DEPTH
        src = [R.pinned_array((S, n * B), np.uint8, write_combined=True) for _ in range(depth)]
        dst = [R.pinned_array((S, pitch), np.int16) for _ in range(depth)]
        for a in src:
            a[...] = iq
        tickets = []

        def go(count):
            for k in range(count):
                if len(tickets) == depth:
                    fb.wait(tickets.pop(0))
                tickets.append(fb.submit(src[k % depth].ctypes.data, n * B, dst[k % depth].ctypes.data, pitch))
            while tickets:
                fb.wait(tickets.pop(0))
        go(depth)
        t0 = time.perf_counter()
        go(steps)
        dt = time.perf_counter() - t0
        for a in src + dst:
            R.free_pinned(a)
    return {"ms_per_call": dt / steps * 1e3, "Gsamples_per_s": S * n * (B // 2) * steps / dt * 1e-9}


def row_in_subprocess(mode, S, n, steps, lib=None):
    """One device-resident row in a fresh process (optionally on another build of the library): a row that fails with
    a stream hand-over time-out is re-run this way on the parent build, to tell a new failure from an old one."""
    env = dict(os.environ)
    env.pop("FMB_LIB_PATH", None)
    if lib:
        env["FMB_LIB_PATH"] = lib
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--only", f"{mode},{S},{n},{steps}"], capture_output=True,
                       text=True, env=env, timeout=300)
    line = [l for l in r.stdout.splitlines() if l.startswith("{")]
    return json.loads(line[-1]) if line else {"error": r.stderr.strip().splitlines()[-1] if r.stderr.strip() else "no output"}


def plan_ab(R, mode, S, n, steps):
    """Kernel 1 time per call under the default rule, tickets of one block each, and the static split."""
    variants = {"default": {}, "one_block_tickets": {"FMB_CHUNK": "8", "FMB_TAIL_PCT": "100"},
                "static_split": {"FMB_CHUNK": "0"}}
    out = {}
    for rep in range(2):                                   # alternated, twice
        for name, env in variants.items():
            for k in ("FMB_CHUNK", "FMB_TAIL_PCT"):
                os.environ.pop(k, None)
            os.environ.update(env)
            try:
                out.setdefault(name, []).append(round(device_rate(R, mode, S, n, steps)["kernel1_ms"], 4))
            except R.FmbError as e:
                out.setdefault(name, []).append(str(e))
    for k in ("FMB_CHUNK", "FMB_TAIL_PCT"):
        os.environ.pop(k, None)
    return out


def bench_ab(parent_tree, reps, steps):
    """bench.py of the parent tree (its own Python binding and library) and of this one, alternated."""
    out = {}
    for rep in range(reps):
        for name, tree in (("parent", parent_tree), ("this", ROOT)):
            for mode in ("stereo", "mono"):
                env = dict(os.environ)
                env.pop("FMB_LIB_PATH", None)
                cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                       "--mode", mode, "--no-cpu", "--no-fma-alt", "--no-other-scaling"]
                r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=tree)
                line = [l for l in r.stdout.splitlines() if l.startswith("{")]
                if r.returncode != 0 or not line:
                    out.setdefault(f"{name}_{mode}", []).append({"error": r.stderr[-500:]})
                    continue
                j = json.loads(line[-1])
                out.setdefault(f"{name}_{mode}", []).append({"value": j["value"], "ms_per_step": j["ms_per_step"],
                                                             "parity": j["parity"]["all"]})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="library built from the parent commit (tools/build_variant.sh): a row that times "
                    "out a stream hand-over wait is re-run on it")
    ap.add_argument("--parent-tree", help="built checkout of the parent commit: its bench.py is the A/B's other arm")
    ap.add_argument("--out", help="JSON file for the results (required unless --only)")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--ab-reps", type=int, default=2)
    ap.add_argument("--sections", default="rates,plan,ab", help="which of rates, plan, ab to run (comma-separated)")
    ap.add_argument("--only", help="mode,streams,blocks,steps: one device-resident row, printed as JSON")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "runs_bench.py measures on a GPU; there is nothing to measure without one"
    if not args.only and not args.out:
        ap.error("--out is required")
    import rtl_fm_player_b200 as R
    if args.only:
        mode, S, n, steps = args.only.split(",")
        try:
            print(json.dumps(device_rate(R, mode, int(S), int(n), int(steps))))
        except R.FmbError as e:
            print(json.dumps({"error": str(e)}))
        return
    sections = set(args.sections.split(","))
    res = {"card": card(), "block_bytes": B, "rates": [], "plan": {}}
    print(res["card"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def save():                                            # after every section: a cut-short run keeps what it measured
        res["card_after"] = card()
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    for mode in ("stereo", "mono") if "rates" in sections else ():
        for S in (1, 8, 64):
            for n in (1, FILL[S]):
                steps = max(4, args.steps // n) if S < 64 else max(4, args.steps // 2)
                row = {"mode": mode, "streams": S, "blocks_per_call": n}
                for k, fn in (("device", device_rate), ("end_to_end", e2e_rate)):
                    try:
                        row[k] = fn(R, mode, S, n, steps)
                    except R.FmbError as e:
                        row[k] = {"error": str(e)}
                if "error" in row["device"]:
                    row["device_fresh_process"] = row_in_subprocess(mode, S, n, steps)
                    if args.parent and os.path.exists(args.parent):
                        row["device_fresh_process_parent_build"] = row_in_subprocess(mode, S, n, steps, args.parent)
                res["rates"].append(row)
                print(json.dumps(row), flush=True)
    save()
    plans = (("stereo", 1024, 2), ("stereo", 64, 4), ("stereo", 8, 16), ("mono", 1024, 2), ("mono", 64, 4))
    for mode, S, n in plans if "plan" in sections else ():
        res["plan"][f"{mode}_{S}x{n}"] = plan_ab(R, mode, S, n, 10)
        print(mode, S, n, res["plan"][f"{mode}_{S}x{n}"], flush=True)
    save()
    if "ab" in sections and args.parent_tree:
        res["bench_ab"] = bench_ab(os.path.abspath(args.parent_tree), args.ab_reps, 20)
        print(json.dumps(res["bench_ab"]), flush=True)
        save()


if __name__ == "__main__":
    main()
