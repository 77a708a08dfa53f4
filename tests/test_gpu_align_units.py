"""Level units of the alignment kernel (DESIGN.md section 4.1): the work queue hands out (pair, level) units instead of
whole pairs.  A pair then runs each level on whichever CTA takes the unit, with the same CTA shape and the same
arithmetic, so every output must be byte-identical to the pair-granular queue.  PLSVO_ALIGN_SCHEDULE forces either mode.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FIELDS = ("T_cur_w", "n_tracked", "H", "seg_killed", "iters", "status", "patch_iters", "patch_levels")
VARIANTS = ["128,4", "256,2"]


def _launch(pkg, data, mode, monkeypatch, levels=(4, 2), variant="128,4", repeat=1):
    monkeypatch.setenv("PLSVO_ALIGN_SCHEDULE", mode)
    monkeypatch.setenv("PLSVO_VARIANT", variant)
    al = pkg.SparseImgAlign(levels[0], levels[1], 30)
    al.upload(data)
    outs = []
    for _ in range(repeat):
        al.launch()
        outs.append(al.download())
    return outs if repeat > 1 else outs[0]


def _same(x, y):
    for f in FIELDS:
        np.testing.assert_array_equal(getattr(x, f), getattr(y, f), err_msg=f)


def _ragged(synth, B, seed, gen_device, n_pts=160, n_segs=40):
    """Ragged per-pair counts, invalid features, empty pairs, points-only and segments-only pairs."""
    data = synth.make_align_batch(batch=B, n_pts=n_pts, n_segs=n_segs, device=gen_device, seed=seed)
    rng = np.random.default_rng(seed)
    data.pt_valid = (rng.uniform(size=(B, n_pts)) > 0.15).astype(np.uint8)
    data.seg_valid = (rng.uniform(size=(B, n_segs)) > 0.15).astype(np.uint8)
    data.pt_count = rng.integers(0, n_pts + 1, B).astype(np.int32)
    data.seg_count = rng.integers(0, n_segs + 1, B).astype(np.int32)
    k = rng.permutation(B)
    data.pt_count[k[0::7]] = 0   # segments only (or empty, with the next line)
    data.seg_count[k[1::7]] = 0  # points only
    data.seg_count[k[0::14]] = 0  # empty pairs
    return data


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("B", [1, 591, 592, 593, 1024, 2048])
def test_level_units_equal_pair_queue(pkg, synth, gen_device, monkeypatch, B, variant):
    data = _ragged(synth, B, 7000 + B, gen_device)
    pair = _launch(pkg, data, "pair", monkeypatch, variant=variant)
    level = _launch(pkg, data, "level", monkeypatch, variant=variant)
    _same(pair, level)
    if B > 1:
        assert (pair.n_tracked == 0).any() and (pair.iters.sum(axis=1) > 0).any()


def test_level_units_points_only(pkg, synth, gen_device, monkeypatch):
    data = synth.make_align_batch(batch=700, n_pts=300, n_segs=0, device=gen_device, seed=7101)
    _same(_launch(pkg, data, "pair", monkeypatch), _launch(pkg, data, "level", monkeypatch))


def test_level_units_segments_only(pkg, synth, gen_device, monkeypatch):
    data = synth.make_align_batch(batch=700, n_pts=0, n_segs=120, device=gen_device, seed=7102)
    _same(_launch(pkg, data, "pair", monkeypatch), _launch(pkg, data, "level", monkeypatch))


@pytest.mark.parametrize("variant", VARIANTS)
def test_level_units_six_levels(pkg, synth, gen_device, monkeypatch, variant):
    """Levels 5 -> 0: six units per pair; the finest level is read through L2, not staged in shared memory."""
    data = synth.make_align_batch(batch=640, n_pts=128, n_segs=32, max_level=5, min_level=0, device=gen_device, seed=7103,
                                  motion_t=0.03, motion_r=0.01)
    pair = _launch(pkg, data, "pair", monkeypatch, levels=(5, 0), variant=variant)
    level = _launch(pkg, data, "level", monkeypatch, levels=(5, 0), variant=variant)
    _same(pair, level)


def test_level_units_back_to_back_launches(pkg, synth, gen_device, monkeypatch):
    """The progress words are tagged with a per-launch epoch and never cleared between launches: a second launch on the
    same batch, and a smaller batch after it, must not see the words the earlier launches left."""
    big = _ragged(synth, 1024, 7104, gen_device)
    small = _ragged(synth, 700, 7105, gen_device)
    ref_big = _launch(pkg, big, "pair", monkeypatch)
    ref_small = _launch(pkg, small, "pair", monkeypatch)
    for out in _launch(pkg, big, "level", monkeypatch, repeat=3):
        _same(ref_big, out)
    for out in _launch(pkg, small, "level", monkeypatch, repeat=2):
        _same(ref_small, out)


def test_level_units_in_track_launch(pkg, synth, gen_device, monkeypatch):
    """plsvo_track_launch: the pose optimiser reads the aligned poses the last unit of each pair writes."""
    al, po = synth.make_track_batch(batch=600, n_pts=300, n_segs=80, seed=7106, device=gen_device)
    res = {}
    for mode in ("pair", "level"):
        monkeypatch.setenv("PLSVO_ALIGN_SCHEDULE", mode)
        monkeypatch.setenv("PLSVO_VARIANT", "128,4")
        res[mode] = pkg.api.track(al, po)
    _same(res["pair"][0], res["level"][0])
    for f in ("T_f_w", "cov", "error_final", "num_obs_pt", "num_obs_ls", "pt_outlier", "seg_outlier", "iters", "status"):
        np.testing.assert_array_equal(getattr(res["pair"][1], f), getattr(res["level"][1], f), err_msg=f)


def test_level_units_oracle_parity_1024_pairs(pkg, abi, synth, oracle, gen_device, monkeypatch):
    """The benchmark's batch (seed 3000, 1024 VGA pairs, levels 4 -> 2), which takes level units by default, against the
    CPU oracle: every pair inside the tolerance and identical integer outputs."""
    monkeypatch.delenv("PLSVO_ALIGN_SCHEDULE", raising=False)
    monkeypatch.delenv("PLSVO_VARIANT", raising=False)
    data = synth.make_align_batch(batch=1024, n_pts=300, n_segs=80, device=gen_device, seed=3000)
    al = pkg.SparseImgAlign(4, 2, 30)
    al.upload(data)
    al.launch()
    gpu = al.download()
    ref = oracle.align(abi, data, n_threads=64)
    ang, rel = synth.pose_error(gpu.T_cur_w, ref.T_cur_w)
    assert ang.max() <= 1e-5 and rel.max() <= 1e-4, (float(ang.max()), float(rel.max()))
    for f in ("iters", "n_tracked", "seg_killed", "status", "patch_levels", "patch_iters"):
        np.testing.assert_array_equal(getattr(gpu, f), getattr(ref, f), err_msg=f)
