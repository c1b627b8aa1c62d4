"""Per-stream output settings: what the per-stream de-emphasis variant costs, and that the uniform path is unchanged.

  * Kernel 2 alone (the de-emphasis + int16 pass, timed by the handle's CUDA-event profile with a device
    synchronisation after every step, as bench.py's pass B does, so that it runs without the next demod launch beside
    it) at 1 024 stereo and 1 024 mono streams, one block per call, and the segmented pass (fmb_deemph_seg_kernel) at
    1 stream x 64 blocks per call.  Four variants, alternated twice:
      uniform    every stream on the handle's own settings (50 us, volume 0.4): the uniform launch;
      volumes    per-stream volumes, de-emphasis as the handle's: the per-stream launch doing the same recurrence work,
                 i.e. the cost of reading the settings from the table;
      mixed      50 us, 75 us, off and 50 us in turn, and per-stream volumes (1 stream: 75 us);
      uniform75  a handle created with 75 us: what the 75 us pole costs by itself (its speculation converges more
                 slowly, so more chunks are redone), to tell that apart from the per-stream launch;
  * the bench.py headlines of a built parent checkout and of this tree, alternated (tools/runs_bench.py bench_ab).
The card's name and power limit are read in the same run.

usage: python tools/stream_output_bench.py --out results.json [--parent-tree DIR] [--sections kernel2,ab]"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from runs_bench import B, bench_ab, card  # noqa: E402  (after the path is set)

DEEMPH = [0.000050, 0.000075, 0.0, 0.000050]
VOLUME = [0.4, 0.7, 0.4, 1.5]
VARIANTS = ("uniform", "volumes", "mixed", "uniform75")


def kernel2(R, mode, S, n, steps, variant):
    import torch
    preset = R.DemodConfig.stereo_192k if mode == "stereo" else R.DemodConfig.mono_192k
    cfg = preset(n_streams=S, max_blocks_per_call=n, deemph=0.000075 if variant == "uniform75" else 0.000050)
    u = min(S, 8)
    kind = "fm_stereo" if mode == "stereo" else "fm_mono"
    iq = np.stack([R.synth.capture(kind, s, 192000, 0, n * B // 2) for s in range(u)])[np.arange(S) % u]
    with R.FmBatch(cfg) as fb:
        vols = np.array(VOLUME * (S // 4 + 1))[:S] if S > 1 else [0.7]
        if variant == "volumes":
            fb.set_stream_output(volume=vols)
        elif variant == "mixed":
            fb.set_stream_output(deemph=np.array(DEEMPH * (S // 4 + 1))[:S] if S > 1 else [0.000075], volume=vols)
        name = fb.deemph_kernel_name()
        pitch = (fb.max_out + 7) & ~7
        d_iq = torch.from_numpy(np.ascontiguousarray(iq)).cuda()
        d_pcm = torch.empty((S, pitch), dtype=torch.int16, device="cuda")
        torch.cuda.synchronize()
        st = R.lib().fmb_internal_stream(fb._h)
        for _ in range(3):
            fb.process_device(d_iq.data_ptr(), n * B, d_pcm.data_ptr(), pitch, st)
        R.lib().fmb_sync(fb._h)
        fb.profile_enable(True)
        fb.profile_reset()
        for _ in range(steps):
            fb.process_device(d_iq.data_ptr(), n * B, d_pcm.data_ptr(), pitch, st)
            R.lib().fmb_sync(fb._h)
        prof = fb.profile_read()
        fallbacks = fb.deemph_fallbacks()
    return {"kernel": name, "kernel2_ms": prof["deemph_ms"] / max(prof["deemph_launches"], 1),
            "launches": prof["deemph_launches"], "fallbacks": fallbacks}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file for the results")
    ap.add_argument("--parent-tree", help="built checkout of the parent commit: its bench.py is the A/B's other arm")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--ab-reps", type=int, default=2)
    ap.add_argument("--sections", default="kernel2,ab", help="which of kernel2, ab to run (comma-separated)")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "stream_output_bench.py measures on a GPU; there is nothing to measure without one"
    import rtl_fm_player_b200 as R
    res = {"card": card(), "block_bytes": B, "kernel2": []}
    print(res["card"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def save():
        res["card_after"] = card()
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    sections = set(args.sections.split(","))
    rows = (("stereo", 1024, 1), ("mono", 1024, 1), ("stereo", 1, 64), ("mono", 1, 64))
    for mode, S, n in rows if "kernel2" in sections else ():
        row = {"mode": mode, "streams": S, "blocks_per_call": n}
        for rep in range(2):
            for v in VARIANTS:
                row.setdefault(v, []).append(kernel2(R, mode, S, n, args.steps, v))
        for v in VARIANTS:
            row[f"{v}_kernel2_ms_median"] = float(np.median([r["kernel2_ms"] for r in row[v]]))
        row["volumes_over_uniform"] = row["volumes_kernel2_ms_median"] / row["uniform_kernel2_ms_median"]
        res["kernel2"].append(row)
        print(json.dumps({k: v for k, v in row.items() if k not in VARIANTS}), flush=True)
        save()
    if "ab" in sections and args.parent_tree:
        res["bench_ab"] = bench_ab(os.path.abspath(args.parent_tree), args.ab_reps, 20)
        print(json.dumps(res["bench_ab"]), flush=True)
    save()


if __name__ == "__main__":
    main()
