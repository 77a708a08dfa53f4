"""Matcher::findMatchDirect (src/matcher.cpp:159-211: affine warp matrix, search level, warped reference patch,
align2D / align1D), SURVEY §8f rank 1.  The oracle restatement is pinned bit for bit against the reference's own
matcher.cpp compiled in place (oracle/_ref); the CUDA kernel must then be bit-identical to the oracle."""
import numpy as np
import pytest

from reference_outputs import Reference


@pytest.mark.parametrize("seed,levels,cam", [(7000, 3, "VGA"), (7001, 5, "VGA"), (7002, 3, "QVGA"), (7003, 4, "HD720")])
def test_oracle_find_match_direct_is_bit_identical_to_the_reference_tu(request, oracle, abi, synth, seed, levels, cam):
    oracle.build_ref()
    d = synth.make_match_batch(cam=getattr(synth, cam), n=1500, seed=seed, n_pyr_levels=levels)
    o = oracle.match_direct(abi, d, 4)
    fields = ("success", "search_level", "px_cur", "A_cur_ref")
    r = Reference(request.node.name, d, lambda: oracle.ref_match_direct(abi, d), fields)
    for f in fields:
        r.assert_equal(f, getattr(o, f))  # A_cur_ref: Matcher::A_cur_ref_ (NaN = untouched on both sides)
    assert np.isfinite(o.A_cur_ref[o.search_level >= 0]).all()
    # the generator plants candidates on the image border: the in-frame test must reject them untouched
    assert (o.search_level < 0).any()
    skipped = o.search_level < 0
    np.testing.assert_array_equal(o.px_cur[skipped], d.px_cur[skipped])
    assert not o.success[skipped].any()


def test_oracle_find_match_direct_refines_towards_the_true_projection(oracle, abi, synth):
    d = synth.make_match_batch(n=1500, seed=7010, edgelet_frac=0.0)
    o = oracle.match_direct(abi, d, 4)
    ok = o.success.astype(bool)
    assert ok.mean() > 0.85
    before = np.abs(d.px_cur - d.px_cur_gt).max(axis=1)
    after = np.abs(o.px_cur - d.px_cur_gt).max(axis=1)
    assert np.median(after[ok]) < 0.35 * np.median(before[ok])


@pytest.mark.gpu
@pytest.mark.parametrize("seed,levels,cam", [(7100, 3, "VGA"), (7101, 5, "VGA"), (7102, 4, "HD720")])
def test_gpu_find_match_direct_is_bit_identical_to_the_oracle(pkg, oracle, abi, synth, gen_device, seed, levels, cam):
    d = synth.make_match_batch(cam=getattr(synth, cam), n=6000, seed=seed, n_pyr_levels=levels, device=gen_device)
    ref = oracle.match_direct(abi, d, 8)
    out = pkg.Matcher(10).findMatchDirect(d)
    np.testing.assert_array_equal(out.search_level, ref.search_level)
    np.testing.assert_array_equal(out.success, ref.success)
    np.testing.assert_array_equal(out.A_cur_ref, ref.A_cur_ref)
    finite = np.isfinite(ref.px_cur).all(axis=1)
    np.testing.assert_array_equal(out.px_cur[finite], ref.px_cur[finite])
    assert (np.isnan(out.px_cur[~finite]) == np.isnan(ref.px_cur[~finite])).all()
    assert ref.success.mean() > 0.5


@pytest.mark.gpu
def test_gpu_find_match_direct_rejects_bad_batches(pkg, abi, synth, gen_device):
    import ctypes as C

    d = synth.make_match_batch(n=64, seed=7200, device=gen_device)
    ctx = pkg.default_context()
    b, keep = abi.make_match_batch(d)
    out = abi.MatchOut(d.n)
    bad = d.ref_index.copy()
    bad[5] = 99
    b.ref_index = bad.ctypes.data_as(C.POINTER(C.c_int32))
    assert ctx.lib.plsvo_match_direct_batch_run(ctx.handle, C.byref(b), C.byref(out.struct)) == abi.ERR_INVALID
    assert b"missing level or frame" in ctx.lib.plsvo_last_error(ctx.handle)
