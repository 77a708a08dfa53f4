"""Structure optimisation — Point::optimize / LineSeg::optimize (src/feature3D_impl.cpp:36-174), SURVEY §8f rank 3.
The oracle restatement is pinned bit for bit against the reference's own feature3D_impl.cpp compiled in place
(oracle/_ref); the CUDA kernel (exact double arithmetic, Eigen's pivoted 3x3 LDLT) must be bit-identical to the oracle."""
import numpy as np
import pytest

from reference_outputs import Reference


@pytest.mark.parametrize("seed,n_iter", [(8000, 5), (8001, 20), (8002, 1), (8003, 0)])
def test_oracle_structopt_is_bit_identical_to_the_reference_tu(request, oracle, abi, synth, seed, n_iter):
    oracle.build_ref()
    d = synth.make_structopt_batch(n_points=1200, n_segs=300, seed=seed)
    d.n_iter_pts = d.n_iter_segs = n_iter
    o = oracle.structopt(abi, d, 4)
    fields = ("pt_pos", "seg_spos", "seg_epos")
    r = Reference(request.node.name, d, lambda: oracle.ref_structopt(abi, d), fields)
    for f in fields:
        r.assert_equal(f, getattr(o, f))
    if n_iter == 0:
        np.testing.assert_array_equal(o.pt_pos, d.pt_pos)


def test_oracle_structopt_moves_points_towards_the_truth(oracle, abi, synth):
    d = synth.make_structopt_batch(n_points=1500, n_segs=300, seed=8010, noise=1e-4)
    o = oracle.structopt(abi, d, 4)
    multi = np.diff(d.pt_obs_begin) >= 3
    before = np.linalg.norm(d.pt_pos - d.pt_pos_gt, axis=1)[multi]
    after = np.linalg.norm(o.pt_pos - d.pt_pos_gt, axis=1)[multi]
    assert np.median(after) < 0.05 * np.median(before)
    sbefore = np.linalg.norm(d.seg_spos - d.seg_spos_gt, axis=1)
    safter = np.linalg.norm(o.seg_spos - d.seg_spos_gt, axis=1)
    assert np.median(safter) < 0.2 * np.median(sbefore)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n_iter", [(8100, 5), (8101, 20), (8102, 1)])
def test_gpu_structopt_is_bit_identical_to_the_oracle(pkg, oracle, abi, synth, seed, n_iter):
    d = synth.make_structopt_batch(n_points=5000, n_segs=1500, seed=seed)
    d.n_iter_pts = d.n_iter_segs = n_iter
    ref = oracle.structopt(abi, d, 8)
    out = pkg.optimizeStructure(d)
    np.testing.assert_array_equal(out.pt_iters, ref.pt_iters)
    np.testing.assert_array_equal(out.seg_iters, ref.seg_iters)
    np.testing.assert_array_equal(out.pt_pos, ref.pt_pos)
    np.testing.assert_array_equal(out.seg_spos, ref.seg_spos)
    np.testing.assert_array_equal(out.seg_epos, ref.seg_epos)


@pytest.mark.gpu
def test_gpu_structopt_points_only_segments_only_and_bad_input(pkg, oracle, abi, synth):
    import ctypes as C

    d = synth.make_structopt_batch(n_points=300, n_segs=0, seed=8200)
    np.testing.assert_array_equal(pkg.optimizeStructure(d).pt_pos, oracle.structopt(abi, d).pt_pos)
    d = synth.make_structopt_batch(n_points=0, n_segs=200, seed=8201)
    np.testing.assert_array_equal(pkg.optimizeStructure(d).seg_epos, oracle.structopt(abi, d).seg_epos)
    d = synth.make_structopt_batch(n_points=50, n_segs=10, seed=8202)
    d.pt_obs_frame = d.pt_obs_frame.copy()
    d.pt_obs_frame[3] = 1000
    ctx = pkg.default_context()
    b, keep = abi.make_structopt_batch(d)
    out = abi.StructOptOut(50, 10)
    assert ctx.lib.plsvo_structopt_batch_run(ctx.handle, C.byref(b), C.byref(out.struct)) == abi.ERR_INVALID


def _structure_case(synth):
    d = synth.make_structopt_batch(n_points=300, n_segs=90, n_frames=9, seed=8123)
    rng = np.random.default_rng(3)
    return d, rng.integers(0, 50, 300).astype(np.int32), rng.integers(0, 50, 90).astype(np.int32)


def _same_structure_result(a, b):
    (oa, pa, sa), (ob, pb, sb) = a, b
    np.testing.assert_array_equal(pa, pb)  # last_structure_optim_: the same features were selected
    np.testing.assert_array_equal(sa, sb)
    np.testing.assert_array_equal(oa.pt_pos, ob.pt_pos)
    np.testing.assert_array_equal(oa.seg_spos, ob.seg_spos)
    np.testing.assert_array_equal(oa.seg_epos, ob.seg_epos)


def test_shim_optimize_structure_packs_reference_objects_like_the_reference_cpu(abi, synth, oracle):
    """plsvo::b200::optimizeStructure (the drop-in body of FrameHandlerBase::optimizeStructure, frame_handler_base.cpp:
    202-237) on the reference's own Point / LineSeg / Frame objects, its C-ABI call answered by the oracle (no GPU):
    same selection, same positions, same last_structure_optim_ as the reference's own loop over Point::optimize."""
    if not oracle.ref_available() or oracle.build_shimref_cpu() is None:
        pytest.skip("oracle/_ref not built and /root/reference absent")
    d, pl, sl = _structure_case(synth)
    ref = oracle.ref_optimize_structure(abi, d, pl, sl, 20, 10)   # Config defaults: structureoptim_max_pts = 20
    got = oracle.shimref_optimize_structure(abi, d, pl, sl, 20, 10, cpu=True)
    _same_structure_result(got, ref)
    assert (got[1] == 77).sum() == 20 and (got[2] == 77).sum() == 10


@pytest.mark.gpu
def test_shim_optimize_structure_on_the_gpu_is_bit_identical_to_the_reference(abi, synth, oracle):
    if not oracle.ref_available() or oracle.build_shimref() is None:
        pytest.skip("oracle/_ref not built and /root/reference absent")
    d, pl, sl = _structure_case(synth)
    for n_pts, n_segs in ((20, 10), (300, 90), (0, 5)):
        ref = oracle.ref_optimize_structure(abi, d, pl, sl, n_pts, n_segs)
        got = oracle.shimref_optimize_structure(abi, d, pl, sl, n_pts, n_segs)
        _same_structure_result(got, ref)
