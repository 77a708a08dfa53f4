#!/usr/bin/env python
"""A/B of the alignment kernel's two work queues in one process: whole pairs (PLSVO_ALIGN_SCHEDULE=pair) against
(pair, level) units (PLSVO_ALIGN_SCHEDULE=level), DESIGN.md section 4.1.

The benchmark's workload (VGA, 300 points + 80 segments per pair, levels 4 -> 2, seed 3000, default CTA shape) at
several batch sizes.  The modes alternate, --rounds times each; every round times --steps launches with CUDA events on
the launch stream and the L2 overwritten (256 MiB write) before each launch, as bench.py does.  The outputs of the two
modes are compared byte for byte.  The card's name and power limit are recorded with the numbers.

usage: python tools/ab_schedule.py [--batches 592,1024,2048,4096] [--rounds 5] [--steps 10] [--out FILE]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FIELDS = ("T_cur_w", "n_tracked", "H", "seg_killed", "iters", "status", "patch_iters", "patch_levels")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="592,1024,2048,4096")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args(argv)

    import torch

    import plsvo_b200
    from plsvo_b200 import synth

    assert torch.cuda.is_available(), "ab_schedule.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = plsvo_b200.Context(0, stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lines = [f"ab_schedule: {card()}; torch {torch.__version__}",
             f"workload: bench.py --config c2 (VGA, 300 pts + 80 segs, levels 4->2, seed 3000), default CTA shape; "
             f"{args.rounds} alternating rounds x {args.steps} launches per mode, L2 flushed before each launch",
             "B      mode   ms/step median [min, max] over rounds     pairs/s (median)   outputs"]
    results = []
    for B in [int(x) for x in args.batches.split(",")]:
        data = synth.make_align_batch(batch=B, n_pts=300, n_segs=80, device=dev, seed=3000)
        al = plsvo_b200.SparseImgAlign(4, 2, 30, ctx=ctx)
        al.upload(data)
        ms = {"pair": [], "level": []}
        outs = {}
        for r in range(args.rounds):
            for mode in ("pair", "level"):
                os.environ["PLSVO_ALIGN_SCHEDULE"] = mode
                al.launch()  # warm-up of this mode
                torch.cuda.synchronize(dev)
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
                for s, e in ev:
                    flush.fill_(1)
                    s.record(stream)
                    al.launch()
                    e.record(stream)
                torch.cuda.synchronize(dev)
                ms[mode].append(sum(s.elapsed_time(e) for s, e in ev) / args.steps)
                if r == 0:
                    outs[mode] = al.download()
        os.environ.pop("PLSVO_ALIGN_SCHEDULE", None)
        same = all(np.array_equal(getattr(outs["pair"], f), getattr(outs["level"], f)) for f in FIELDS)
        row = {"B": B}
        for mode in ("pair", "level"):
            v = np.array(ms[mode])
            med = float(np.median(v))
            row[mode] = {"ms_median": med, "ms_min": float(v.min()), "ms_max": float(v.max()), "ms_rounds": [round(x, 4) for x in v]}
            lines.append(f"{B:<6} {mode:<6} {med:.4f} [{v.min():.4f}, {v.max():.4f}]{'':14} {B / med * 1e3:,.0f}"
                         f"{'':8} {'byte-identical' if same else 'DIFFER'}")
        gain = row["pair"]["ms_median"] / row["level"]["ms_median"] - 1
        lines.append(f"{B:<6} level vs pair: {100 * gain:+.1f} % pairs/s")
        row["identical"] = same
        results.append(row)
    text = "\n".join(lines)
    print(text)
    print(json.dumps(results))
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    return 0 if all(r["identical"] for r in results) else 1


if __name__ == "__main__":
    sys.exit(main())
