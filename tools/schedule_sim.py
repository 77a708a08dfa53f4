#!/usr/bin/env python
"""Predict what handing out (pair, level) units instead of whole pairs does to the alignment kernel's makespan.

A CPU model of the persistent grid's work queue (DESIGN.md section 4.1).  Inputs are the benchmark batch's per-pair,
per-level Gauss-Newton pass counts and per-level patch counts:
  * pass counts: from a `bench.py --dump-outputs DIR` file (iters.npy) or, without one, from the CPU oracle on the
    benchmark's seeded inputs (synth.make_align_batch(seed=3000));
  * patch counts: from the same seeded inputs, computed the way the kernel sets them up (points inside the level's
    border, segment samples 1 + (N0 - 1) >> level of segments whose endpoints are inside).
A unit costs passes x patches + a set-up term (the reference-patch precompute: about one pass over the patches, plus a
fixed part).  The queue is list-scheduled onto the grid's slots: in pair order for the pair queue, level-major for
level units, where a unit cannot start before the same pair's unit at the level above has finished.  Times are in
patch-pass units; only the ratio of the two makespans is meant to be read.

usage: python tools/schedule_sim.py [--dump DIR] [--batch 1024] [--slots 592] [--setup-fixed 200] [--out FILE]"""
from __future__ import annotations

import argparse
import heapq
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)


def patch_counts(data, levels):
    """[B, n_levels] patches set up per pair and level (points inside the border, segment samples)."""
    W, H = data.cam.width, data.cam.height
    B = data.batch
    out = np.zeros((B, len(levels)), np.int64)
    spx, epx, length = data.seg_spx, data.seg_epx, data.seg_length
    d = np.abs(epx - spx)
    with np.errstate(divide="ignore", invalid="ignore"):
        tan_dir = np.minimum(d[..., 0], d[..., 1]) / np.maximum(d[..., 0], d[..., 1])
    sin_dir = tan_dir / np.sqrt(1.0 + tan_dir * tan_dir)
    nd = length / (8.0 * 2.0 * np.sqrt(1.0 + sin_dir * sin_dir))
    nd = np.where(nd >= 1.0, nd, 1.0)
    N0 = np.minimum(nd, 1048576.0).astype(np.int64)
    for k, l in enumerate(levels):
        cols, rows, s = W >> l, H >> l, 1.0 / (1 << l)

        def inside(px, border, c=cols, r=rows):
            u = np.floor(px[..., 0] * s)
            v = np.floor(px[..., 1] * s)
            return (u >= border) & (v >= border) & (u < c - border) & (v < r - border)

        n_pts = inside(data.pt_px, 3).sum(axis=1)
        seg_in = inside(spx, 3) & inside(epx, 3)
        n_samples = np.where(seg_in, 1 + ((N0 - 1) >> l), 0).sum(axis=1)
        out[:, k] = n_pts + n_samples
    return out


def makespan(costs, order, slots, dep):
    """List scheduling: the next ticket goes to the slot that frees first; a ticket with a dependency starts no earlier
    than that ticket's finish (the slot waits)."""
    free = [0.0] * slots
    heapq.heapify(free)
    finish = {}
    end = 0.0
    for t in order:
        s = heapq.heappop(free)
        start = max(s, finish.get(dep(t), 0.0)) if dep(t) is not None else s
        f = start + costs[t]
        finish[t] = f
        end = max(end, f)
        heapq.heappush(free, f)
    return end


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--dump", default="", help="bench.py --dump-outputs directory (iters.npy); default: run the oracle")
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--slots", type=int, default=592, help="resident CTAs of the grid (148 SMs x 4 for <128,4>)")
    ap.add_argument("--setup-fixed", type=float, default=200.0, help="fixed part of a unit's set-up, in patch-passes")
    ap.add_argument("--max-level", type=int, default=4)
    ap.add_argument("--min-level", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args(argv)

    from plsvo_b200 import abi, synth

    levels = list(range(args.max_level, args.min_level - 1, -1))
    data = synth.make_align_batch(batch=args.batch, n_pts=300, n_segs=80, seed=3000)
    if args.dump:
        iters = np.load(os.path.join(args.dump, "iters.npy")).astype(np.int64)
        source = f"pass counts from {os.path.basename(os.path.normpath(args.dump))}/iters.npy"
    else:
        import oracle_lib

        oracle_lib.build()
        iters = oracle_lib.align(abi, data, abi.align_params(args.max_level, args.min_level, 30), n_threads=os.cpu_count()).iters
        source = "pass counts from the CPU oracle"
    iters = iters[:, levels]
    patches = patch_counts(data, levels)
    unit = iters * patches + patches + args.setup_fixed  # [B, n_levels]
    B, nl = unit.shape

    pair_cost = unit.sum(axis=1)
    t_pair = makespan(pair_cost, range(B), args.slots, lambda t: None)
    flat = unit.T.reshape(-1)  # ticket k*B + b = pair b at level index k
    t_level = makespan(flat, range(B * nl), args.slots, lambda t: t - B if t >= B else None)
    ideal = unit.sum() / args.slots
    lines = [
        f"schedule_sim: B={B} pairs, {args.slots} slots, levels {args.max_level}->{args.min_level}; {source}",
        f"unit cost = passes x patches + patches (precompute) + {args.setup_fixed:g}",
        f"passes per level (mean): " + ", ".join(f"L{l} {iters[:, k].mean():.2f}" for k, l in enumerate(levels)),
        f"patches per level (mean): " + ", ".join(f"L{l} {patches[:, k].mean():.1f}" for k, l in enumerate(levels)),
        f"pair cost: mean {pair_cost.mean():.0f}, min {pair_cost.min():.0f}, max {pair_cost.max():.0f}",
        f"work / slots (no idle slot, lower bound): {ideal:.0f}",
        f"pair queue makespan       : {t_pair:.0f}  ({t_pair / ideal:.3f} x bound)",
        f"level-unit queue makespan : {t_level:.0f}  ({t_level / ideal:.3f} x bound)",
        f"predicted step time ratio level/pair: {t_level / t_pair:.3f}  (gain {100 * (t_pair / t_level - 1):.1f} % in pairs/s)",
        "caveat: slots are modelled as independent; on the GPU the resident CTAs of an SM share its issue rate, so a CTA "
        "left alone on an SM runs faster and the pair queue's idle tail costs less than modelled: read the gain as an "
        "upper estimate",
    ]
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
