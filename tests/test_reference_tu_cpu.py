"""Pins the oracle restatement against THE REFERENCE ITSELF, run here.

oracle/_ref/libplsvo_ref.so is the reference's own src/sparse_img_align.cpp, src/pose_optimizer.cpp and
src/feature.cpp, compiled unmodified from /root/reference against the reference's own headers and
stand-in third-party headers (oracle/refdeps, oracle/ref_harness.cpp).  The oracle
(oracle/plsvo_oracle.cpp) must reproduce it BIT FOR BIT on every output the ABI carries — poses, H,
n_tracked, killed segments, per-level iteration counts, status; pose, covariance, scale, errors,
observation counts and outlier flags for the pose optimiser — over the edge cases the domain has
(empty / ragged / masked feature lists, borders, zero motion, large motion, long segments, 720p).

The library is built by __graft_entry__.build() / oracle_lib.build_ref() where the original sources are; elsewhere
the tests compare with the record of its outputs (tests/reference_outputs.py).
"""
import numpy as np
import pytest

from reference_outputs import Reference


@pytest.fixture(scope="module")
def ref(oracle, abi):
    if oracle.build_ref():
        oracle.load_ref(abi)
    return oracle


ALIGN_FIELDS = ("T_cur_w", "n_tracked", "H", "seg_killed", "iters", "status")
PO_FIELDS = ("T_f_w", "cov", "estimated_scale", "error_init", "error_final", "num_obs_pt", "num_obs_ls", "pt_outlier",
             "seg_outlier", "status")


def assert_align_identical(key, ref, abi, data, params=None, threads=4):
    a = ref.align(abi, data, params, n_threads=threads)
    r = Reference(key, (data, params), lambda: ref.ref_align(abi, data, params, n_threads=threads), ALIGN_FIELDS)
    for f in ALIGN_FIELDS:
        r.assert_equal(f, getattr(a, f))
    return a


def assert_poseopt_identical(key, ref, abi, data, params):
    a = ref.poseopt(abi, data, params, n_threads=2)
    r = Reference(key, (data, params), lambda: ref.ref_poseopt(abi, data, params, n_threads=2), PO_FIELDS)
    for f in PO_FIELDS:
        r.assert_equal(f, getattr(a, f))
    return a


@pytest.mark.parametrize("cfg", [
    dict(cam="QVGA", batch=12, n_pts=120, n_segs=30, seed=101),
    dict(cam="VGA", batch=8, n_pts=300, n_segs=80, seed=102),                       # BASELINE config C2 shape
    dict(cam="VGA", batch=6, n_pts=300, n_segs=0, seed=103),                        # points only
    dict(cam="VGA", batch=6, n_pts=0, n_segs=80, seed=104),                         # segments only
    dict(cam="VGA", batch=6, n_pts=200, n_segs=60, seed=105, margin=6),             # features at the image border
    dict(cam="VGA", batch=6, n_pts=200, n_segs=60, seed=106, motion_t=0.15, motion_r=0.05),  # large motion: rollbacks
    dict(cam="HD720", batch=3, n_pts=300, n_segs=80, seed=107),
    dict(cam="HD720", batch=2, n_pts=500, n_segs=150, seed=109),                    # BASELINE config 4 shape
    dict(cam="QVGA", batch=6, n_pts=64, n_segs=16, seed=108, max_level=3, min_level=0),       # down to level 0
])
def test_align_restatement_is_bit_identical_to_reference_tus(request, ref, abi, synth, cfg):
    cfg = dict(cfg)
    cfg["cam"] = getattr(synth, cfg["cam"])
    data = synth.make_align_batch(**cfg)
    out = assert_align_identical(request.node.name, ref, abi, data)
    if cfg["n_pts"]:
        assert (out.n_tracked > 0).all()


def test_align_ragged_masked_and_empty_pairs(request, ref, abi, synth):
    data = synth.make_align_batch(cam=synth.QVGA, batch=12, n_pts=96, n_segs=40, seed=110)
    rng = np.random.default_rng(5)
    data.pt_valid = (rng.uniform(size=(12, 96)) > 0.2).astype(np.uint8)
    data.seg_valid = (rng.uniform(size=(12, 40)) > 0.2).astype(np.uint8)
    data.pt_count = rng.integers(1, 97, 12).astype(np.int32)
    data.seg_count = rng.integers(0, 41, 12).astype(np.int32)
    data.pt_count[3] = 0
    data.seg_count[3] = 0  # empty pair: run() returns 0 and leaves the pose untouched (sparse_img_align.cpp:58-62)
    data.pt_count[5] = 0   # segments only
    data.seg_count[7] = 0  # points only
    data.pt_valid[9] = 0
    data.seg_valid[9] = 0  # features present but every feat3D == NULL
    out = assert_align_identical(request.node.name, ref, abi, data)
    assert out.status[3] & 1 and out.n_tracked[3] == 0
    np.testing.assert_array_equal(out.T_cur_w[3], data.T_cur_w[3])


def test_align_zero_motion_raises_stop_like_the_reference(request, ref, abi, synth):
    """cur == ref: every residual is 0, the per-segment mean residual is 0 and H_*weight/res_ divides by it
    (sparse_img_align.cpp:676): the solve returns NaN and vk::NLLSSolver raises stop_."""
    data = synth.make_align_batch(cam=synth.QVGA, batch=3, n_pts=64, n_segs=16, seed=111, motion_t=0.0, motion_r=0.0)
    out = assert_align_identical(request.node.name, ref, abi, data)
    assert (out.status & 2).all()


def test_align_long_segments_and_iteration_limits(request, ref, abi, synth):
    """Segments spanning the image (many 4x4 samples each, some samples leaving the frame -> killed segments),
    at levels 2..0, and tight iteration / level limits."""
    import torch

    data = synth.make_align_batch(cam=synth.VGA, batch=4, n_pts=80, n_segs=12, max_level=2, min_level=0, seed=112,
                                  motion_t=0.004, motion_r=0.0012, margin=24)
    rng = np.random.default_rng(3)
    B, S = data.seg_spx.shape[:2]
    spx = np.stack([rng.uniform(30, 150, (B, S)), rng.uniform(30, 450, (B, S))], -1)
    epx = np.stack([rng.uniform(480, 610, (B, S)), rng.uniform(30, 450, (B, S))], -1)
    scene = synth.Scene()
    R, t = synth.pose7_to_Rt(torch.tensor(data.T_ref_w))

    def lift(px):
        p = torch.tensor(px)
        d = torch.stack([(p[..., 0] - data.cam.cx) / data.cam.fx, (p[..., 1] - data.cam.cy) / data.cam.fy, torch.ones_like(p[..., 0])], -1)
        f = d / d.norm(dim=-1, keepdim=True)
        return f.numpy(), scene.intersect(R, t, d).numpy()

    data.seg_spx, data.seg_epx = np.ascontiguousarray(spx), np.ascontiguousarray(epx)
    data.seg_sf, data.seg_spos = (np.ascontiguousarray(x) for x in lift(spx))
    data.seg_ef, data.seg_epos = (np.ascontiguousarray(x) for x in lift(epx))
    data.seg_length = np.ascontiguousarray(np.linalg.norm(epx - spx, axis=-1))
    key = request.node.name
    assert_align_identical(key + "/2-0", ref, abi, data, abi.align_params(2, 0, 30))
    assert_align_identical(key + "/2-1", ref, abi, data, abi.align_params(2, 1, 3))   # n_iter = 3
    assert_align_identical(key + "/2-2", ref, abi, data, abi.align_params(2, 2, 30))  # a single level


@pytest.mark.parametrize("n_ref", [-1, 0, 5])
@pytest.mark.parametrize("cfg", [
    dict(batch=24, seed=201),
    dict(batch=12, seed=202, n_segs=0),
    dict(batch=12, seed=203, outlier_frac=0.35),
    dict(batch=12, seed=204, noise_px=2.0, pert_t=0.08, pert_r=0.04),
    dict(batch=12, seed=205, noise_px=0.0, outlier_frac=0.0),
])
def test_poseopt_restatement_is_bit_identical_to_reference_tus(request, ref, abi, synth, cfg, n_ref):
    data = synth.make_poseopt_batch(**cfg)
    assert_poseopt_identical(request.node.name, ref, abi, data, abi.poseopt_params(2.0, 10, n_ref))


def test_poseopt_ragged_and_masked(request, ref, abi, synth):
    data = synth.make_poseopt_batch(batch=10, n_pts=64, n_segs=24, seed=210)
    rng = np.random.default_rng(9)
    data.pt_valid = (rng.uniform(size=(10, 64)) > 0.25).astype(np.uint8)
    data.seg_valid = (rng.uniform(size=(10, 24)) > 0.25).astype(np.uint8)
    data.pt_count = rng.integers(8, 65, 10).astype(np.int32)
    data.seg_count = rng.integers(0, 25, 10).astype(np.int32)
    data.pt_valid[2] = 0
    data.seg_valid[2] = 0  # no observations at all: early return (pose_optimizer.cpp:88-89)
    for n_ref in (-1, 4):
        out = assert_poseopt_identical(f"{request.node.name}/{n_ref}", ref, abi, data, abi.poseopt_params(2.0, 10, n_ref))
        assert out.status[2] == 1
        np.testing.assert_array_equal(out.T_f_w[2], data.T_f_w[2])


def test_golden_fixtures_are_reference_outputs(request, ref, abi, synth):
    """tests/golden/*.npz were written from oracle/_ref (tests/golden/make_golden.py): what the reference's own code
    computes on their inputs must be the committed vectors bit for bit."""
    from golden_io import load_align, load_poseopt

    d, z = load_align(synth)
    p = abi.align_params(3, 1, 30)
    fields = ("T_cur_w", "n_tracked", "H", "seg_killed", "iters")
    r = Reference(request.node.name + "/align", (d, p), lambda: ref.ref_align(abi, d, p), fields)
    assert "sparse_img_align" in str(z["source"])
    for f in fields:
        r.assert_equal(f, z[f"out_{f}"])
    d, z = load_poseopt(synth)
    fields = ("T_f_w", "cov", "estimated_scale", "error_init", "error_final", "num_obs_pt", "num_obs_ls", "pt_outlier",
              "seg_outlier")
    for tag, n_ref in (("9arg", -1), ("10arg", 3)):
        p = abi.poseopt_params(2.0, 10, n_ref)
        r = Reference(f"{request.node.name}/{tag}", (d, p), lambda: ref.ref_poseopt(abi, d, p), fields)
        for f in fields:
            r.assert_equal(f, z[f"out_{tag}_{f}"], err_msg=f"{tag} {f}")


def test_shim_packs_reference_objects_like_the_reference_reads_them(ref, abi, synth):
    """pl-svo_b200/host/plsvo_shim.cpp compiled in -DPLSVO_SHIM_WITH_REFERENCE_HEADERS mode, fed with the reference's own
    Frame / PointFeat / LineFeat / Point / LineSeg objects, with the C ABI answered by the CPU oracle (oracle/abi_on_oracle.cpp,
    test infrastructure): what comes back in those objects must be what the reference's own sparse_img_align.cpp /
    pose_optimizer.cpp leave in them.  (The GPU run of the same harness is tests/test_gpu_shim.py.)"""
    if not ref.build_shimref_cpu():
        pytest.skip("needs /root/reference")
    d = synth.make_align_batch(cam=synth.QVGA, batch=8, n_pts=120, n_segs=30, seed=120)
    d.seg_valid = np.ones((8, 30), np.uint8)
    d.seg_valid[:, ::5] = 0
    d.pt_valid = np.ones((8, 120), np.uint8)
    d.pt_valid[:, ::9] = 0
    got = ref.shimref_align(abi, d, cpu=True)
    want = ref.ref_align(abi, d)
    np.testing.assert_array_equal(got.n_tracked, want.n_tracked)
    np.testing.assert_array_equal(got.seg_killed, want.seg_killed)
    # poses make one extra trip through SE3's quaternion normalisation on the way in and out: last-bit differences only
    np.testing.assert_allclose(got.T_cur_w, want.T_cur_w, rtol=0, atol=1e-12)
    np.testing.assert_allclose(got.H * (5e-4 * 255 * 255), want.H, rtol=1e-9, atol=1e-9 * np.abs(want.H).max())
    pd = synth.make_poseopt_batch(batch=8, n_pts=100, n_segs=30, seed=121)
    for n_ref in (-1, 3):
        p = abi.poseopt_params(2.0, 10, n_ref)
        got, want = ref.shimref_poseopt(abi, pd, p, cpu=True), ref.ref_poseopt(abi, pd, p)
        for f in ("num_obs_pt", "num_obs_ls", "pt_outlier", "seg_outlier"):
            np.testing.assert_array_equal(getattr(got, f), getattr(want, f), err_msg=f)
        np.testing.assert_allclose(got.T_f_w, want.T_f_w, rtol=0, atol=1e-12)
        np.testing.assert_allclose(got.cov, want.cov, rtol=1e-9, atol=1e-15)
        for f in ("estimated_scale", "error_init", "error_final"):
            np.testing.assert_allclose(getattr(got, f), getattr(want, f), rtol=1e-12, err_msg=f)


def test_sequence_chain_oracle_equals_reference_chain(request, abi, synth, oracle):
    """BASELINE config 1 on the CPU: frame-to-frame chain (align -> pose-opt, the estimate seeds the next frame,
    frame_handler_mono.cpp:263-340) over short QVGA sequences — the oracle restatement and the reference's own
    translation units give bit-identical poses, iteration counts and outlier flags at every frame, and the chain tracks
    the ground-truth trajectory."""
    if oracle.build_ref():
        oracle.load_ref(abi)
    poses, steps = synth.make_sequence(cam=synth.QVGA, n_seq=2, n_frames=6, n_pts=120, n_segs=30, seed=1000)

    def chain(align_fn, po_fn):
        def step(al, po):
            ra = align_fn(abi, al, abi.align_params(al.max_level, al.min_level, 30), n_threads=4)
            po.T_f_w = np.ascontiguousarray(ra.T_cur_w)
            return ra, po_fn(abi, po, abi.poseopt_params(2.0, 10, -1), n_threads=4)
        return synth.run_sequence(poses, steps, step)

    r = Reference(request.node.name, (poses, steps),
                  lambda: dict(zip(("est", "iters", "outliers"), chain(oracle.ref_align, oracle.ref_poseopt))))
    est_o, it_o, out_o = chain(oracle.align, oracle.poseopt)
    r.assert_equal("est", est_o)
    r.assert_equal("iters", it_o)
    r.assert_equal("outliers", out_o)
    ang, rel = synth.pose_error(est_o[:, -1], poses[:, -1])
    assert ang.max() < 1e-2
