#!/usr/bin/env python
"""bench.py — frame-pair aligns/s of the B200-native PL-SVO alignment path (BASELINE.json metric).

A "step" is one pass of the hot path (plsvo::SparseImgAlign::run, coarse-to-fine levels 4->2,
<=30 GN iterations per level) over one batch of synthetic frame pairs: VGA, 5-level pyramid,
300 point patches + 80 line segments per pair.  Per-GPU work is fixed (weak scaling): every rank
aligns its own batch, no data-path collective; poses are gathered with one NCCL all_gather.

  value      : pairs/s, inputs resident in HBM, kernel time from CUDA events on the launch stream
  e2e        : pairs/s through the C-ABI call with pinned HOST buffers (H2D + kernel + D2H timed)
  roofline   : algorithmic bytes (241 B per patch-iteration + 281 B per patch-level, SURVEY.md §8d)
               / kernel time, against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline: the reference's CPU implementation on this box's host cores — oracle/_ref (the
               reference's own sparse_img_align.cpp/feature.cpp compiled against stand-in third-party
               headers, kind "reference") when that library was built, else the oracle restatement ("port")

`--impl reference` times that CPU implementation alone (rank 0), same metric/config.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "frame-pair aligns/sec (VGA 5-lvl pyr, ~300pt+80ln)"
BYTES_PATCH_ITER = 241
BYTES_PATCH_LEVEL = 281
BYTES_PAIR_FIXED = 512
DTYPE = "f32 residuals, weights and chi2 (the reference's summation order, bit-exact); f64 per-pixel normal equations, solve and SE3"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="frame pairs per GPU per step")
    ap.add_argument("--n-pts", type=int, default=300)
    ap.add_argument("--n-segs", type=int, default=80)
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs per CPU-baseline pass (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="device-resident leg only, compact output (tuning)")
    ap.add_argument("--no-next", action="store_true", help="skip the SURVEY 8f (next-row) kernel block of the line")
    ap.add_argument("--no-chain", action="store_true", help="skip the frame-chain end-to-end leg (e2e_chain)")
    ap.add_argument("--config", default="c2", choices=["c2", "c4"],
                    help="c2: BASELINE configs[1] + the metric's 80 lines (headline); c4: configs[3], chained align -> pose-opt at 720p")
    ap.add_argument("--sweep", action="store_true", help="BASELINE configs[4]: patch count x pyramid depth sweep (JSON list)")
    ap.add_argument("--sweep-out", default="", help="also write the sweep's JSON to this file (rank 0)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step of the device-resident leg returned as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "c4" or args.sweep):
        ap.error("--dump-outputs is for the alignment leg (--config c2, --impl b200, no --sweep)")
    return args


DUMP_LIMIT = 64_000_000 - (1 << 16)  # bytes of array data: at most 64 MB written, with room left for the .npy headers
DUMP_FIELDS = ("T_cur_w", "n_tracked", "H", "seg_killed", "iters", "status", "patch_iters", "patch_levels")


def dump_outputs(out, directory):
    """SparseImgAlign::run's outputs per pair as float64 .npy files (integer outputs are exact in float64).  A batch
    whose outputs exceed DUMP_LIMIT is written as a fixed, seeded sample of pairs, listed in pair_index.npy."""
    arrays = {n: np.asarray(getattr(out, n)).astype(np.float64) for n in DUMP_FIELDS}
    B = len(arrays["T_cur_w"])
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    if B * row_bytes > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_LIMIT // (row_bytes + 8), replace=False))
        arrays = {n: a[keep] for n, a in arrays.items()}
        arrays["pair_index"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(directory, n + ".npy"), a)


def workload_config(args, n_gpus):
    return {
        "workload": "SparseImgAlign::run, VGA 640x480, 5-level pyramid (levels 4->2 used), "
                    f"{args.n_pts} point patches + {args.n_segs} line segments per pair, <=30 GN iters/level",
        "pairs_per_gpu_per_step": args.batch,
        "global_batch": args.batch * n_gpus,
        "parallelism": f"dp{n_gpus} (independent frame pairs, no data-path collective)",
        "l2": "flushed between timed steps (256 MiB write)",
    }


class ClockSampler:
    """nvidia-smi clock/throttle sampling during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.check_output(
                    ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                    timeout=5).decode().strip()
                self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_source_hash():
    """sha256 over the alignment kernel's sources (align_kernel.cu, device_math.cuh, the AlignArgs block of internal.h): ties a committed ncu traffic capture to the code it measured."""
    import hashlib

    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "pl-svo_b200", "csrc")
    for f in ("align_kernel.cu", "device_math.cuh"):
        h.update(open(os.path.join(csrc, f), "rb").read())
    # internal.h: only the alignment kernel's argument block (everything before the first separator line; the other
    # kernels' argument structs follow it and do not enter this kernel)
    head = open(os.path.join(csrc, "internal.h"), "rb").read().split(b"\n// -----", 1)[0]
    h.update(head)
    return h.hexdigest()


def committed_traffic(args):
    """DRAM bytes per launch of sparse_img_align_kernel from the committed `ncu --set full` capture of this exact
    configuration — only if that capture was taken from the kernel source that is being timed now."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["sparse_img_align_kernel"]
    except Exception:
        return None, "no committed capture (profiles/r02_traffic.json)"
    if not (args.batch == tj.get("batch") and args.n_pts == tj.get("n_pts") and args.n_segs == tj.get("n_segs")):
        return None, "committed capture is for another configuration"
    if tj.get("kernel_source_sha256") != kernel_source_hash():
        return None, "STALE: kernel source changed since the committed capture " + str(tj.get("source"))
    return tj["dram_bytes_per_launch"], tj["source"]


def cpu_impl(abi, oracle_lib):
    """(align function, kind, description) of the CPU arm: oracle/_ref when built, else the oracle port."""
    if oracle_lib.ref_available():
        return (oracle_lib.ref_align, "reference",
                "oracle/_ref: the reference's own src/sparse_img_align.cpp + feature.cpp compiled unmodified against "
                "stand-in Eigen/Sophus/vikit/OpenCV headers (oracle/refdeps), -O3")
    return (oracle_lib.align, "port",
            "oracle restatement of sparse_img_align.cpp (oracle/_ref not built on this box)")


def subset(data, n_pairs):
    """The first n_pairs of an AlignData batch (copies)."""
    import copy

    sub = copy.copy(data)
    sl = slice(0, n_pairs)
    for name in ("T_ref_w", "T_cur_w", "T_cur_w_gt", "pt_px", "pt_f", "pt_pos", "seg_spx", "seg_epx", "seg_sf", "seg_ef",
                 "seg_spos", "seg_epos", "seg_length"):
        setattr(sub, name, np.ascontiguousarray(getattr(data, name)[sl]))
    sub.ref_pyr = {l: np.ascontiguousarray(v[sl]) for l, v in data.ref_pyr.items()}
    sub.cur_pyr = {l: np.ascontiguousarray(v[sl]) for l, v in data.cur_pyr.items()}
    return sub


def lean_copy(data, torch):
    """What the end-to-end leg ships: the finest level used only (coarser levels are halfSample'd on the device), the
    distance of every 3-D feature from the reference camera centre instead of its position, and no bearing vectors (they
    are cam2world(px) for the undistorted pinhole camera; include/plsvo_b200.h).
    Returns (AlignData, bytes, keepalive); every array is pinned."""
    import copy

    from plsvo_b200 import synth

    lean = copy.copy(data)
    R, t = synth.pose7_to_Rt(torch.tensor(data.T_ref_w))
    centre = -(R.transpose(1, 2) @ t[..., None])[..., 0].numpy()  # Frame::pos(), frame.h:131
    lean.pt_depth = np.ascontiguousarray(np.linalg.norm(data.pt_pos - centre[:, None, :], axis=-1))
    lean.seg_sdepth = np.ascontiguousarray(np.linalg.norm(data.seg_spos - centre[:, None, :], axis=-1))
    lean.seg_edepth = np.ascontiguousarray(np.linalg.norm(data.seg_epos - centre[:, None, :], axis=-1))
    lean.pt_pos = lean.seg_spos = lean.seg_epos = None
    lean.pt_f = lean.seg_sf = lean.seg_ef = None  # undistorted pinhole: cam2world(px) on the device (feature.cpp:42,98-99)
    lean.ref_pyr = {data.min_level: data.ref_pyr[data.min_level]}
    lean.cur_pyr = {data.min_level: data.cur_pyr[data.min_level]}
    keep, nbytes = [], 0
    for name in ("T_ref_w", "T_cur_w", "pt_px", "pt_depth", "seg_spx", "seg_epx", "seg_sdepth", "seg_edepth", "seg_length"):
        tt = torch.from_numpy(getattr(lean, name)).pin_memory()
        setattr(lean, name, tt.numpy())
        keep.append(tt)
        nbytes += tt.numpy().nbytes
    for pyr in (lean.ref_pyr, lean.cur_pyr):
        for l in list(pyr):
            tt = torch.from_numpy(pyr[l]).pin_memory()
            pyr[l] = tt.numpy()
            keep.append(tt)
            nbytes += tt.numpy().nbytes
    return lean, nbytes, keep


def chain_leg(args, al, synth, torch, dev, stream, B, rank):
    """The local part of the `e2e_chain` leg: B pairs replaying one trajectory of B + 1 frames, shipped as two stacks once
    (the comparison) and then as one stack (PLSVO_ALIGN_FRAME_CHAIN), warm-up + args.steps timed calls from page-locked
    arrays.  Returns (ms over the timed calls, (full batch, last result, H2D bytes per call, check against the two-stack
    call)).  Kept free of collectives so that the caller can wrap it in a try; tests/hostmodel/scenarios.py runs it against
    the host model."""
    cfull = synth.make_chain_batch(batch=B, n_pts=args.n_pts, n_segs=args.n_segs, device=dev, seed=7000 + 100000 * rank)
    clean, _h2d_two, keep_chain = lean_copy(cfull, torch)
    two = al.run(clean)  # the same chain given as two stacks (ref, cur): the comparison for the one-stack call
    ft = torch.from_numpy(synth.chain_frames(cfull, levels=[cfull.min_level])[cfull.min_level]).pin_memory()
    keep_chain.append(ft)
    clean.frame_pyr = {cfull.min_level: ft.numpy()}
    h2d_chain = (_h2d_two - sum(v.nbytes for v in clean.ref_pyr.values()) - sum(v.nbytes for v in clean.cur_pyr.values())
                 + ft.numpy().nbytes)
    for _ in range(2):
        out_c = al.run(clean)
    _a, _r = synth.pose_error(out_c.T_cur_w, two.T_cur_w)
    chain_check = {"iteration_counts_equal_to_two_stack_call": int((out_c.iters == two.iters).all(axis=1).sum()), "pairs": int(B),
                   "max_rot_rad_vs_two_stack_call": float(_a.max()), "max_rel_t_vs_two_stack_call": float(_r.max())}
    torch.cuda.synchronize(dev)
    c_s, c_e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    c_s.record(stream)
    for _ in range(args.steps):
        out_c = al.run(clean)
    c_e.record(stream)
    torch.cuda.synchronize(dev)
    chain_local_ms = max(c_s.elapsed_time(c_e), 1e3 * (time.perf_counter() - t0))
    return chain_local_ms, (cfull, out_c, h2d_chain, chain_check)


def cpu_oracle_rate(abi, oracle_lib, data, n_pairs, min_seconds=3.0):
    """pairs/s of the CPU arm with all host threads on the first n_pairs of `data`."""
    align_fn, _, _ = cpu_impl(abi, oracle_lib)
    sub = subset(data, n_pairs)
    hw = max(1, oracle_lib.load(abi).plsvo_oracle_hardware_threads())
    # the box may expose more logical CPUs than it lets us run on: take the best of a few thread counts
    best = None
    for threads in sorted({hw, max(1, hw // 2), max(1, hw // 4), max(1, hw // 8)}, reverse=True):
        align_fn(abi, sub, n_threads=threads)  # warm
        t0 = time.perf_counter()
        align_fn(abi, sub, n_threads=threads)
        r = n_pairs / (time.perf_counter() - t0)
        if best is None or r > best[0]:
            best = (r, threads)
    threads = best[1]
    t0 = time.perf_counter()
    reps = 0
    while True:
        align_fn(abi, sub, n_threads=threads)
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            break
    return reps * n_pairs / dt, threads, dt, reps


def _events(torch, stream, n):
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]


def poseopt_alg_bytes(pout, n_pts, n_segs):
    """SURVEY 8d: 52 B per (point, pass) + 76 B per (line, pass); passes = MAD + executed GN iterations + outlier pass."""
    passes = 2.0 + pout.iters[:, 0].astype(np.float64)
    return float((passes * (52 * n_pts + 76 * n_segs)).sum())


def run_c4(args, rank, world, local_rank):
    """BASELINE configs[3]: combined align + pose path, 720p 5-level pyramid, 500 points + 150 lines, batch sharded across
    the GPUs.  One step = SparseImgAlign::run followed by pose_optimizer::optimizeGaussNewton on every frame of the
    rank's batch, the pose staying on the device in between (plsvo_track_*)."""
    import ctypes as C

    import torch

    import plsvo_b200
    from plsvo_b200 import abi, synth

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    B = args.batch
    n_pts, n_segs = (500, 150) if (args.n_pts, args.n_segs) == (300, 80) else (args.n_pts, args.n_segs)
    al, po = synth.make_track_batch(cam=synth.HD720, batch=B, n_pts=n_pts, n_segs=n_segs, seed=3000 + 100000 * rank, device=dev)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = plsvo_b200.Context(local_rank, stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ap, pp = abi.align_params(4, 2, 30), abi.poseopt_params(2.0, 10, -1)
    ab, keep_a = abi.make_align_batch(al)
    pb, keep_p = abi.make_poseopt_batch(po)
    pb.T_f_w = abi._f64p()  # chained: start from the aligned pose on the device
    ao, pout = abi.AlignOut(B, n_segs), abi.PoseOptOut(B, n_pts, n_segs)
    L = ctx.lib
    ctx.check(L.plsvo_track_upload(ctx.handle, C.byref(ab), C.byref(pb)), "track upload")
    for _ in range(args.warmup):
        ctx.check(L.plsvo_track_launch(ctx.handle, C.byref(ap), C.byref(pp)), "track launch")
    ctx.sync()
    launches0 = ctx.launch_count()
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    clk = ClockSampler(local_rank)
    clk.__enter__()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    for s0, s1, s2 in ev:
        flush.fill_(1)
        s0.record(stream)
        ctx.check(L.plsvo_align_launch(ctx.handle, C.byref(ap)), "align launch")
        s1.record(stream)
        ctx.check(L.plsvo_poseopt_launch(ctx.handle, C.byref(pp)), "poseopt launch")  # reads the aligned poses on the device
        s2.record(stream)
    torch.cuda.synchronize(dev)
    launches = ctx.launch_count() - launches0
    al_ms = [a.elapsed_time(b) for a, b, _ in ev]
    po_ms = [b.elapsed_time(c) for _, b, c in ev]
    total_ms = float(sum(a.elapsed_time(c) for a, _, c in ev))
    ctx.check(L.plsvo_align_download(ctx.handle, C.byref(ao.struct)), "align download")
    ctx.check(L.plsvo_poseopt_download(ctx.handle, C.byref(pout.struct)), "poseopt download")
    t_total = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if dist:
        from plsvo_b200 import dist as pdist

        all_poses = pdist.gather_rows(pout.T_f_w, world * B, device=dev)
        assert all_poses.shape == (world * B, 7)
        dist.all_reduce(t_total, op=dist.ReduceOp.MAX)
        dist.barrier()
    torch.cuda.synchronize(dev)
    max_ms = float(t_total.item())
    value = world * B * args.steps / (max_ms * 1e-3)
    # ---- end to end through the chained C-ABI call, pinned host buffers in, host results out ----
    pins = []
    for obj, names in ((al, ("T_ref_w", "T_cur_w", "pt_px", "pt_f", "pt_pos", "seg_spx", "seg_epx", "seg_sf", "seg_ef", "seg_spos",
                             "seg_epos", "seg_length")),
                       (po, ("pt_f", "pt_pos", "pt_level", "seg_line", "seg_spos", "seg_epos", "seg_level"))):
        for name in names:
            tt = torch.from_numpy(getattr(obj, name)).pin_memory()
            setattr(obj, name, tt.numpy())
            pins.append(tt)
    lean, h2d_al, keep_l = lean_copy(al, torch)
    h2d = h2d_al + sum(getattr(po, n).nbytes for n in ("pt_f", "pt_pos", "pt_level", "seg_line", "seg_spos", "seg_epos", "seg_level"))
    for _ in range(2):
        ao_e, po_e = plsvo_b200.api.track(lean, po, ctx=ctx)
    c4_e2e_check = {"align_iteration_counts_equal_to_device_leg": int((ao_e.iters == ao.iters).all(axis=1).sum()), "frames": int(B),
                    "outlier_flags_equal_to_device_leg": bool(np.array_equal(po_e.pt_outlier, pout.pt_outlier))}
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ao_e, po_e = plsvo_b200.api.track(lean, po, ctx=ctx)
    torch.cuda.synchronize(dev)
    e2e_ms = torch.tensor([1e3 * (time.perf_counter() - t0)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    clk.__exit__(None, None, None)
    e2e_value = world * B * args.steps / (float(e2e_ms.item()) * 1e-3)
    d2h = sum(getattr(ao_e, n).nbytes for n in ("T_cur_w", "n_tracked", "H", "seg_killed", "iters", "status", "patch_iters", "patch_levels"))
    d2h += sum(getattr(po_e, n).nbytes for n in ("T_f_w", "cov", "estimated_scale", "error_init", "error_final", "num_obs_pt",
                                                 "num_obs_ls", "pt_outlier", "seg_outlier", "iters", "status"))
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        al_bytes = float(ao.patch_iters.astype(np.float64).sum() * BYTES_PATCH_ITER
                         + ao.patch_levels.astype(np.float64).sum() * BYTES_PATCH_LEVEL + B * BYTES_PAIR_FIXED)
        po_bytes = poseopt_alg_bytes(pout, n_pts, n_segs)
        al_s, po_s = float(np.mean(al_ms)) * 1e-3, float(np.mean(po_ms)) * 1e-3
        cpu = None
        if not args.no_cpu_baseline:
            import copy

            import oracle_lib

            n = min(args.cpu_sample or 256, B)
            sub = subset(al, n)
            have_ref = oracle_lib.ref_available()
            align_fn = oracle_lib.ref_align if have_ref else oracle_lib.align
            po_fn = oracle_lib.ref_poseopt if have_ref else oracle_lib.poseopt
            hw = max(1, oracle_lib.load(abi).plsvo_oracle_hardware_threads())
            threads = max(1, min(64, hw // 2))
            psub = copy.copy(po)
            for name in ("T_f_w", "T_f_w_gt", "pt_f", "pt_pos", "pt_level", "seg_line", "seg_spos", "seg_epos", "seg_level"):
                setattr(psub, name, np.ascontiguousarray(getattr(po, name)[:n]))

            def chain():
                ra = align_fn(abi, sub, n_threads=threads)
                psub.T_f_w = np.ascontiguousarray(ra.T_cur_w)
                return ra, po_fn(abi, psub, abi.poseopt_params(2.0, 10, -1), n_threads=threads)

            chain()
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 3.0:
                ra, rp = chain()
                reps += 1
            dt = time.perf_counter() - t0
            ang, rel = synth.pose_error(pout.T_f_w[:n], rp.T_f_w)
            cpu = {"value": reps * n / dt, "unit": "frames/s", "cores": threads, "kind": "reference" if have_ref else "port",
                   "sample": f"{n} frames x {reps} passes ({dt:.1f} s): SparseImgAlign::run then optimizeGaussNewton from its result, "
                             f"{threads} host threads",
                   "parity_vs_gpu": {"max_rot_rad": float(ang.max()), "max_rel_t": float(rel.max()),
                                     "frames_within_tol": int(((ang <= 1e-5) & (rel <= 1e-4)).sum()), "frames": n,
                                     "align_iteration_counts_equal": int((ao.iters[:n] == ra.iters).all(axis=1).sum()),
                                     "outlier_flags_equal": bool(np.array_equal(pout.pt_outlier[:n], rp.pt_outlier)
                                                                 and np.array_equal(pout.seg_outlier[:n], rp.seg_outlier))}}
        line = {
            "metric": "frames/s through align + pose-opt (720p 5-lvl pyr, 500pt+150ln), chained on the device",
            "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic",
            "config": {"workload": f"BASELINE configs[3]: SparseImgAlign::run (levels 4->2, <=30 GN iters/level) then "
                                   f"pose_optimizer::optimizeGaussNewton (<=10 iters) from the aligned pose, 1280x720, "
                                   f"{n_pts} points + {n_segs} line segments per frame", "frames_per_gpu_per_step": B,
                       "global_batch": B * world, "parallelism": f"dp{world} (independent frames, no data-path collective)",
                       "l2": "flushed between timed steps (256 MiB write)"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(d2h) * world,
                    "check": c4_e2e_check},
            "gpu_launches": int(launches), "clocks": clk.summary(),
            "roofline": {"bound": "hbm", "kernel": "sparse_img_align_kernel", "achieved": al_bytes / al_s / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": al_bytes / al_s / 1e9 / peak, "traffic": None,
                         "traffic_source": "not captured for this configuration", "peak_source": peak_src,
                         "avg_kernel_ms": al_s * 1e3, "share_of_step": al_s / (al_s + po_s),
                         "second_kernel": {"kernel": "pose_optimizer_kernel", "avg_kernel_ms": po_s * 1e3,
                                           "achieved": po_bytes / po_s / 1e9, "frac": po_bytes / po_s / 1e9 / peak}},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()
    return 0


SWEEP_N = (64, 128, 256, 512, 1024, 2048)
SWEEP_L = (3, 4, 5, 6)


def run_sweep(args, rank, world, local_rank):
    """BASELINE configs[4]: patch count 64 -> 2048 x pyramid depth 3 -> 6 (max_level = L-1, min_level = max(L-3, 0): the
    reference's three-level schedule, SURVEY 8d C5), every cell with pairs/s, the algorithmic roofline fraction, parity
    against the CPU arm on a sample and that arm's rate.  Under torchrun every rank runs its own batches (weak scaling)."""
    import torch

    import plsvo_b200
    from plsvo_b200 import abi, synth

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = plsvo_b200.Context(local_rank, stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    peak, _ = measured_hbm_peak()
    cells = []
    import oracle_lib

    have_ref = oracle_lib.ref_available()
    align_fn = oracle_lib.ref_align if have_ref else oracle_lib.align
    hw = max(1, oracle_lib.load(abi).plsvo_oracle_hardware_threads())
    threads = max(1, min(64, hw // 2))
    for L in SWEEP_L:
        max_level, min_level = L - 1, max(L - 3, 0)
        for N in SWEEP_N:
            n_segs = int(round(N * 80 / 300))
            B = args.batch if N <= 512 else max(148, args.batch // (N // 512 * 2))
            shrink = 1 << max(0, 4 - max_level)
            data = synth.make_align_batch(batch=B, n_pts=N, n_segs=n_segs, max_level=max_level, min_level=min_level,
                                          seed=7000 + 17 * N + L + 100000 * rank, device=dev, motion_t=0.03 / shrink, motion_r=0.01 / shrink)
            al = plsvo_b200.SparseImgAlign(max_level, min_level, 30, ctx=ctx)
            cell = {"n_pts": N, "n_segs": n_segs, "pyramid_levels": L, "max_level": max_level, "min_level": min_level, "pairs_per_gpu": B}
            try:
                al.upload(data)
                for _ in range(2):
                    al.launch()
                ctx.sync()
                ts = []
                for _ in range(max(3, args.steps // 2)):
                    flush.fill_(1)
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record(stream)
                    al.launch()
                    e.record(stream)
                    torch.cuda.synchronize(dev)
                    ts.append(s.elapsed_time(e))
                out = al.download()
                ms = float(np.median(ts))
                t = torch.tensor([ms], dtype=torch.float64, device=dev)
                if dist:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_max = float(t.item())
                alg = float(out.patch_iters.astype(np.float64).sum() * BYTES_PATCH_ITER
                            + out.patch_levels.astype(np.float64).sum() * BYTES_PATCH_LEVEL + B * BYTES_PAIR_FIXED)
                cell.update({"ms_per_step": ms_max, "pairs_per_s": world * B / (ms_max * 1e-3), "algorithmic_GBps": alg / (ms * 1e-3) / 1e9,
                             "roofline_frac": alg / (ms * 1e-3) / 1e9 / peak, "mean_gn_passes": float(out.iters.sum(axis=1).mean()),
                             "status_flags": int((out.status >> 2).astype(bool).sum())})
                if rank == 0:
                    n = min(96 if N <= 512 else 48, B)
                    sub = subset(data, n)
                    align_fn(abi, sub, n_threads=threads)
                    t0 = time.perf_counter()
                    ref = align_fn(abi, sub, n_threads=threads)
                    dt = time.perf_counter() - t0
                    ang, rel = synth.pose_error(out.T_cur_w[:n], ref.T_cur_w)
                    cell["cpu"] = {"pairs_per_s": n / dt, "threads": threads, "kind": "reference" if have_ref else "port", "pairs": n}
                    cell["parity"] = {"pairs": n, "within_tol": int(((ang <= 1e-5) & (rel <= 1e-4)).sum()),
                                      "iteration_counts_equal": int((out.iters[:n] == ref.iters).all(axis=1).sum()),
                                      "max_rot_rad": float(ang.max()), "max_rel_t": float(rel.max())}
            except Exception as ex:
                cell["error"] = str(ex)
            cells.append(cell)
            if rank == 0:
                print(json.dumps(cell), file=sys.stderr, flush=True)
            del data, al
    if rank == 0:
        doc = {"sweep": "BASELINE configs[4]: patch count x pyramid depth", "n_gpus": world, "unit": "pairs/s",
               "peak_GBps": peak, "cells": cells}
        print(json.dumps(doc))
        if args.sweep_out:
            json.dump(doc, open(args.sweep_out, "w"), indent=1)
    if dist:
        dist.destroy_process_group()
    return 0


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = max(world, 1)

    import plsvo_b200
    from plsvo_b200 import abi, synth

    if args.impl != "reference" and args.sweep:
        return run_sweep(args, rank, world, local_rank)
    if args.impl != "reference" and args.config == "c4":
        return run_c4(args, rank, world, local_rank)
    if args.impl == "reference":
        if rank != 0:
            return 0
        import oracle_lib
        import torch

        n = args.cpu_sample or args.batch
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        data = synth.make_align_batch(batch=n, n_pts=args.n_pts, n_segs=args.n_segs, device=dev, seed=3000)
        align_fn, kind, what = cpu_impl(abi, oracle_lib)
        hw = max(1, oracle_lib.load(abi).plsvo_oracle_hardware_threads())
        best = None  # logical CPUs may exceed what the box lets us run on: pick the fastest thread count
        for th in sorted({hw, max(1, hw // 2), max(1, hw // 4), max(1, hw // 8)}, reverse=True):
            align_fn(abi, data, n_threads=th)
            t0 = time.perf_counter()
            align_fn(abi, data, n_threads=th)
            r = n / (time.perf_counter() - t0)
            if best is None or r > best[0]:
                best = (r, th)
        threads = best[1]
        for _ in range(args.warmup):
            align_fn(abi, data, n_threads=threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            align_fn(abi, data, n_threads=threads)
        dt = time.perf_counter() - t0
        val = args.steps * n / dt
        cfg = workload_config(args, n_gpus)
        line = {
            "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": threads, "kind": kind,
                             "sample": f"{n} pairs per step x {args.steps} steps; {what}"},
            "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return 0

    import torch

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    B = args.batch
    data = synth.make_align_batch(batch=B, n_pts=args.n_pts, n_segs=args.n_segs, device=dev, seed=3000 + 100000 * rank)

    # every rank runs on the CPUs of its own GPU's NUMA node while it allocates and fills its page-locked buffers and drives
    # the GPU legs (plsvo_b200.numa); the affinity is handed back before any CPU arm is timed
    from plsvo_b200 import numa

    placement = numa.describe(local_rank)
    saved_affinity = numa.bind_to_device(local_rank)
    placement["bound"] = saved_affinity is not None

    # pinned host copies of every input array (the e2e leg copies from these every step)
    def pin(a):
        t = torch.from_numpy(a).pin_memory()
        return t.numpy(), t

    keep = []
    for name in ("T_ref_w", "T_cur_w", "pt_px", "pt_f", "pt_pos", "seg_spx", "seg_epx", "seg_sf", "seg_ef", "seg_spos",
                 "seg_epos", "seg_length"):
        arr, t = pin(getattr(data, name))
        setattr(data, name, arr)
        keep.append(t)
    for pyr in (data.ref_pyr, data.cur_pyr):
        for l in list(pyr):
            arr, t = pin(pyr[l])
            pyr[l] = arr
            keep.append(t)
    h2d = sum(getattr(data, n).nbytes for n in ("T_ref_w", "T_cur_w", "pt_px", "pt_f", "pt_pos", "seg_spx", "seg_epx", "seg_sf",
                                                "seg_ef", "seg_spos", "seg_epos", "seg_length"))
    h2d += sum(v.nbytes for v in data.ref_pyr.values()) + sum(v.nbytes for v in data.cur_pyr.values())

    # a non-default torch stream, handed to the C ABI so that torch.cuda.Event sees the kernels
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx = plsvo_b200.Context(local_rank, stream.cuda_stream)
    al = plsvo_b200.SparseImgAlign(4, 2, 30, plsvo_b200.SparseImgAlign.GaussNewton, False, False, ctx=ctx)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # ---- device-resident leg ----
    al.upload(data)
    for _ in range(args.warmup):
        al.launch()
    ctx.sync()
    out0 = al.download()
    d2h = sum(getattr(out0, n).nbytes for n in ("T_cur_w", "n_tracked", "H", "seg_killed", "iters", "status", "patch_iters",
                                                "patch_levels"))
    launches0 = ctx.launch_count()
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    clk = ClockSampler(local_rank)
    clk.__enter__()  # sampled over both timed legs (device-resident and end-to-end)
    for s, e in ev:
        flush.fill_(1)  # evict the batch from L2 (outside the timed events)
        s.record(stream)
        al.launch()
        e.record(stream)
    torch.cuda.synchronize(dev)
    kernel_ms = [s.elapsed_time(e) for s, e in ev]
    launches = ctx.launch_count() - launches0
    total_ms = float(sum(kernel_ms))
    out = al.download()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    t_total = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if dist:
        from plsvo_b200 import dist as pdist

        all_poses = pdist.gather_rows(out.T_cur_w, world * B, device=dev)  # gather poses (NCCL all_gather)
        assert all_poses.shape == (world * B, 7)
        dist.all_reduce(t_total, op=dist.ReduceOp.MAX)
        dist.barrier()
    torch.cuda.synchronize(dev)
    max_ms = float(t_total.item())
    value = n_gpus * B * args.steps / (max_ms * 1e-3)

    if args.quick:
        clk.__exit__(None, None, None)
        if rank == 0:
            print(json.dumps({"quick": True, "value": value, "ms_per_step": max_ms / args.steps,
                              "kernel_ms": [round(x, 4) for x in kernel_ms],
                              "lib": os.environ.get("PLSVO_LIB", "default"),
                              "env": {k: v for k, v in os.environ.items() if k.startswith("PLSVO_")}}))
        if dist:
            dist.destroy_process_group()
        return 0

    # ---- end-to-end leg: pinned host buffers -> C ABI -> host results, every step ----
    # ships what the reference-facing call needs at minimum (lean_copy): finest used level + feature depths
    data_full = data
    data, h2d, keep_lean = lean_copy(data_full, torch)
    for _ in range(2):
        out_e2e = al.run(data)
    # the lean inputs must give the device-resident leg's result: recorded in the line, not asserted (a last-bit
    # difference of a derived bearing may legitimately move a pose by ~1e-9)
    _a, _r = synth.pose_error(out_e2e.T_cur_w, out.T_cur_w)
    e2e_check = {"iteration_counts_equal_to_device_leg": int((out_e2e.iters == out.iters).all(axis=1).sum()), "pairs": int(B),
                 "max_rot_rad_vs_device_leg": float(_a.max()), "max_rel_t_vs_device_leg": float(_r.max())}
    data_lean = data
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e_s, e_e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e_s.record(stream)
    for _ in range(args.steps):
        out_e2e = al.run(data)
    e_e.record(stream)
    torch.cuda.synchronize(dev)
    e2e_wall = time.perf_counter() - t0
    e2e_ms = torch.tensor([max(e_s.elapsed_time(e_e), 1e3 * e2e_wall)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = n_gpus * B * args.steps / (float(e2e_ms.item()) * 1e-3)
    clk.__exit__(None, None, None)
    data = data_full
    numa.restore(saved_affinity)  # the CPU arms below get every host thread back

    # ---- multi-GPU product path: ONE host batch on rank 0 -> NCCL scatter -> align on every GPU -> all_gather ----
    e2e_scatter = None
    if dist:
        from plsvo_b200 import dist as pdist

        glob = None
        if rank == 0:
            import copy

            glob = copy.copy(data_lean)  # rank 0's lean batch, tiled: world x B pairs owned by one process
            for name in pdist._ALIGN_ARRAYS:
                a = getattr(data_lean, name, None)
                if a is not None:
                    setattr(glob, name, np.concatenate([a] * world, 0))
            glob.ref_pyr = {l: np.concatenate([v] * world, 0) for l, v in data_lean.ref_pyr.items()}
            glob.cur_pyr = {l: np.concatenate([v] * world, 0) for l, v in data_lean.cur_pyr.items()}
        pdist.align_sharded(glob, 4, 2, 30, src=0, device=dev, ctx=ctx)  # warm
        dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        n_sc = 2
        for _ in range(n_sc):
            full = pdist.align_sharded(glob, 4, 2, 30, src=0, device=dev, ctx=ctx)
        torch.cuda.synchronize(dev)
        sc_ms = torch.tensor([1e3 * (time.perf_counter() - t0) / n_sc], dtype=torch.float64, device=dev)
        dist.all_reduce(sc_ms, op=dist.ReduceOp.MAX)
        assert full["T_cur_w"].shape == (world * B, 7)
        sharded_same = bool(np.array_equal(full["iters"][:B], out.iters)) if rank == 0 else None
        e2e_scatter = {"value": world * B / (float(sc_ms.item()) * 1e-3), "unit": "pairs/s", "ms_per_step": float(sc_ms.item()),
                       "iteration_counts_equal_to_device_leg": sharded_same,
                       "what": "plsvo_b200.dist.align_sharded: one host batch of n_gpus x %d pairs on rank 0 (rank 0's batch tiled), "
                               "packed per shard, NCCL scatter, align on every GPU, all_gather of all outputs; timed wall clock "
                               "including the Python-side packing" % B}

    # ---- roofline of the alignment kernel (the only kernel in the step) ----
    alg_bytes = float(out.patch_iters.astype(np.float64).sum() * BYTES_PATCH_ITER
                      + out.patch_levels.astype(np.float64).sum() * BYTES_PATCH_LEVEL + B * BYTES_PAIR_FIXED)
    avg_kernel_s = (total_ms / args.steps) * 1e-3
    peak, peak_src = measured_hbm_peak()
    achieved = alg_bytes / avg_kernel_s / 1e9
    traffic, traffic_src = committed_traffic(args)

    # ---- secondary: pose optimiser (BASELINE config 3: 300 pts + 80 lines, 10 iters, B = 4096 frames) ----
    poseopt = None
    try:
        pdata = synth.make_poseopt_batch(batch=4096, n_pts=args.n_pts, n_segs=args.n_segs, seed=5000 + rank)
        # page-locked host arrays, as for the alignment legs (the end-to-end call copies straight from them)
        ppin, p_h2d = [], 0
        for name in ("T_f_w", "pt_f", "pt_pos", "pt_level", "seg_line", "seg_spos", "seg_epos", "seg_level"):
            tt = torch.from_numpy(np.ascontiguousarray(getattr(pdata, name))).pin_memory()
            setattr(pdata, name, tt.numpy())
            ppin.append(tt)
            p_h2d += tt.numpy().nbytes
        pbatch, pkeep = abi.make_poseopt_batch(pdata)
        pout = abi.PoseOptOut(pdata.batch, pdata.n_pts, pdata.n_segs)
        pparams = abi.poseopt_params(2.0, 10, -1)
        import ctypes as C

        ctx.check(ctx.lib.plsvo_poseopt_upload(ctx.handle, C.byref(pbatch)), "poseopt upload")
        for _ in range(3):
            ctx.check(ctx.lib.plsvo_poseopt_launch(ctx.handle, C.byref(pparams)), "poseopt launch")
        torch.cuda.synchronize(dev)
        pts = []
        for _ in range(5):
            flush.fill_(1)
            s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s_.record(stream)
            ctx.check(ctx.lib.plsvo_poseopt_launch(ctx.handle, C.byref(pparams)), "poseopt launch")
            e_.record(stream)
            torch.cuda.synchronize(dev)
            pts.append(s_.elapsed_time(e_))
        ctx.check(ctx.lib.plsvo_poseopt_download(ctx.handle, C.byref(pout.struct)), "poseopt download")
        pms = float(np.median(pts))
        pbytes = poseopt_alg_bytes(pout, pdata.n_pts, pdata.n_segs)
        # end to end through the host-buffer call, and the CPU arm with parity on the same frames (rank 0)
        ctx.check(ctx.lib.plsvo_poseopt_batch_run(ctx.handle, C.byref(pbatch), C.byref(pparams), C.byref(pout.struct)), "poseopt run")
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(5):
            ctx.check(ctx.lib.plsvo_poseopt_batch_run(ctx.handle, C.byref(pbatch), C.byref(pparams), C.byref(pout.struct)), "poseopt run")
        pe2e = 5 * pdata.batch / (time.perf_counter() - t0)
        p_d2h = sum(getattr(pout, n).nbytes for n in ("T_f_w", "cov", "estimated_scale", "error_init", "error_final", "num_obs_pt",
                                                      "num_obs_ls", "pt_outlier", "seg_outlier", "iters", "status") if hasattr(pout, n))
        pcpu = None
        if rank == 0 and not args.no_cpu_baseline:
            import oracle_lib

            have_ref = oracle_lib.ref_available()
            pfn = oracle_lib.ref_poseopt if have_ref else oracle_lib.poseopt
            hw = max(1, oracle_lib.load(abi).plsvo_oracle_hardware_threads())
            pth = max(1, min(64, hw // 2))
            pfn(abi, pdata, pparams, n_threads=pth)
            t0 = time.perf_counter()
            pref = pfn(abi, pdata, pparams, n_threads=pth)
            pdt = time.perf_counter() - t0
            pang, prel = synth.pose_error(pout.T_f_w, pref.T_f_w)
            pcpu = {"value": pdata.batch / pdt, "unit": "frames/s", "cores": pth, "kind": "reference" if have_ref else "port",
                    "sample": f"{pdata.batch} frames, one pass",
                    "parity_vs_gpu": {"max_rot_rad": float(pang.max()), "max_rel_t": float(prel.max()),
                                      "frames_within_tol": int(((pang <= 1e-5) & (prel <= 1e-4)).sum()), "frames": int(pdata.batch),
                                      "outlier_flags_equal": bool(np.array_equal(pout.pt_outlier, pref.pt_outlier)
                                                                  and np.array_equal(pout.seg_outlier, pref.seg_outlier))}}
        poseopt = {"metric": "pose-optimiser frames/s (300 pts + 80 lines, <=10 GN iters, B=4096)",
                   "value": pdata.batch / (pms * 1e-3), "unit": "frames/s", "ms_per_batch": pms,
                   "note": "includes the per-launch clearing of 6 small output arrays (memsets)",
                   "e2e": {"value": pe2e, "unit": "frames/s", "h2d_bytes_per_step": int(p_h2d), "d2h_bytes_per_step": int(p_d2h),
                           "note": "plsvo_poseopt_batch_run from page-locked host arrays, results to host (wall clock over 5 calls)"},
                   "cpu_baseline": pcpu,
                   "roofline": {"bound": "hbm", "achieved": pbytes / (pms * 1e-3) / 1e9, "unit": "GB/s",
                                "frac": pbytes / (pms * 1e-3) / 1e9 / measured_hbm_peak()[0]}}
    except Exception as ex:  # secondary number: never take the headline line down
        poseopt = {"error": str(ex)}

    # ---- SURVEY 8f next-row kernels (N = 1 only): kernel rate, host-in/host-out rate from pinned memory, CPU oracle beside
    # them on all host threads, exactness against it on the timed inputs (tools/bench_next.py holds the full accounting) ----
    next_rows = None
    if rank == 0 and n_gpus == 1 and not args.no_next and not args.no_cpu_baseline:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_next

            nr = bench_next.measure(reps=5, images=64, features=100000, struct_points=50000, ctx=ctx, dev=dev)
            next_rows = {"host_memory": nr.get("host_memory"), "detail": "python tools/bench_next.py (full sizes) -> profiles/r02_next_kernels.json"}
            for name, row in nr.items():
                if not isinstance(row, dict):
                    continue
                k = next((x for x in row if x.endswith("_per_s_kernel")), None)
                unit = k[: -len("_per_s_kernel")] + "/s"
                exact = next((row[x] for x in row if "exact" in x), None)
                next_rows[name] = {"unit": unit, "kernel": row[k], "e2e": row[k.replace("_kernel", "_e2e")],
                                   "cpu": next(row[x] for x in row if x.startswith("cpu_oracle_")), "cpu_threads": row["cpu_threads"],
                                   "exact_vs_oracle": exact, "workload": row["workload"]}
        except Exception as ex:  # secondary block: never take the headline line down
            next_rows = {"error": repr(ex)}

    # ---- end-to-end leg on a frame chain: the same call replaying ONE trajectory of B + 1 frames (pair b = frames b, b+1;
    # src/frame_handler_mono.cpp:176,272) shipped as one stack, PLSVO_ALIGN_FRAME_CHAIN — every frame crosses the link once.
    # Single-process run only, and after every other leg that touches the GPU: this is the youngest host path and its leg had
    # not been timed on hardware when it was added, so nothing else in the line depends on its outcome, and the lines under
    # torchrun keep exactly the legs they were measured with ----
    e2e_chain = None
    if not args.no_chain and not dist:
        rebound = numa.bind_to_device(local_rank)  # as for the e2e leg
        try:
            chain_local_ms, chain_info = chain_leg(args, al, synth, torch, dev, stream, B, rank)
            e2e_chain = {"value": B * args.steps / (chain_local_ms * 1e-3), "unit": "pairs/s",
                         "h2d_bytes_per_step": int(chain_info[2]), "d2h_bytes_per_step": int(d2h), "check": chain_info[3],
                         "workload": "same call and feature mix on a frame chain: %d pairs replaying one trajectory of %d frames, "
                                     "frames shipped once as one stack (PLSVO_ALIGN_FRAME_CHAIN)" % (B, B + 1),
                         "_cpu_inputs": chain_info[:2]}
        except Exception as ex:  # secondary leg: never take the headline line down
            e2e_chain = {"error": f"{type(ex).__name__}: {ex}"}
        numa.restore(rebound)

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            import oracle_lib

            n = args.cpu_sample or B
            rate, threads, secs, reps = cpu_oracle_rate(abi, oracle_lib, data, min(n, B))
            # parity of the timed batch against the CPU arm on the same inputs
            ref = cpu_impl(abi, oracle_lib)[0](abi, data, n_threads=threads)
            ang, rel = synth.pose_error(out.T_cur_w, ref.T_cur_w)
            _, kind, what = cpu_impl(abi, oracle_lib)
            # SURVEY 8d(i): the reference's own call pattern, one pair at a time on one thread
            n1 = min(48, B)
            sub1 = subset(data, n1)
            cpu_impl(abi, oracle_lib)[0](abi, sub1, n_threads=1)
            t1 = time.perf_counter()
            cpu_impl(abi, oracle_lib)[0](abi, sub1, n_threads=1)
            single = n1 / (time.perf_counter() - t1)
            cpu = {"value": rate, "unit": "pairs/s", "cores": threads, "kind": kind,
                   "single_thread": {"value": single, "unit": "pairs/s", "cores": 1, "ms_per_pair": 1e3 / single, "pairs": n1},
                   "iteration_counts_equal": int((out.iters == ref.iters).all(axis=1).sum()),
                   "sample": f"{min(n, B)} pairs x {reps} passes ({secs:.1f} s), all host threads; {what}",
                   "parity_vs_gpu": {"max_rot_rad": float(ang.max()), "max_rel_t": float(rel.max()),
                                     "pairs_within_tol": int(((ang <= 1e-5) & (rel <= 1e-4)).sum()), "pairs": int(B)}}
        if e2e_chain and "_cpu_inputs" in e2e_chain:
            cin = e2e_chain.pop("_cpu_inputs")
            if cin is not None and not args.no_cpu_baseline:
                try:  # secondary leg: a failure of its checker is recorded, the headline line still goes out
                    import oracle_lib

                    n_c = min(128, B)  # bounded sample: the first pairs of the chain against the CPU arm
                    ref_c = cpu_impl(abi, oracle_lib)[0](abi, subset(cin[0], n_c), n_threads=cpu["cores"] if cpu else 8)
                    ang_c, rel_c = synth.pose_error(cin[1].T_cur_w[:n_c], ref_c.T_cur_w)
                    e2e_chain["parity_vs_cpu"] = {"pairs": int(n_c), "pairs_within_tol": int(((ang_c <= 1e-5) & (rel_c <= 1e-4)).sum()),
                                                  "iteration_counts_equal": int((cin[1].iters[:n_c] == ref_c.iters).all(axis=1).sum()),
                                                  "max_rot_rad": float(ang_c.max()), "max_rel_t": float(rel_c.max())}
                except Exception as ex:
                    e2e_chain["parity_vs_cpu"] = {"error": f"{type(ex).__name__}: {ex}"}
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic", "config": workload_config(args, n_gpus),
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d) * n_gpus,
                    "d2h_bytes_per_step": int(d2h) * n_gpus, "check": e2e_check},
            "e2e_chain": e2e_chain,
            "e2e_scatter": e2e_scatter,
            "host_placement": placement,
            "gpu_launches": int(launches),
            "clocks": clk.summary(),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": "sparse_img_align_kernel",
                         "algorithmic_bytes_per_launch": alg_bytes, "avg_kernel_ms": total_ms / args.steps,
                         "mean_gn_passes_per_pair": float(out.iters.sum(axis=1).mean())},
            "cpu_baseline": cpu,
            "poseopt": poseopt,
            "next_rows": next_rows,
        }
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
