"""Depth-filter point-seed update (DepthFilter::updatePointSeeds body, Matcher::findEpipolarMatchDirect, computeTau,
updatePointSeed; src/depth_filter.cpp:270-365,489-512,568-584, src/matcher.cpp:277-420), SURVEY §8f rank 4.

CPU: the oracle restatement reproduces the reference's own depth_filter.cpp + matcher.cpp (compiled in place,
oracle/_ref) bit for bit.  GPU: status, search result and triangulated depth are bit-identical to the oracle; the
updated seed agrees to float round-off, because computeTau and the Gaussian pdf go through acos / sin / atan / expf,
whose last bit differs between glibc and the CUDA math library (tolerances stated below)."""
import numpy as np
import pytest

from reference_outputs import Reference

SEED_FIELDS = ("status", "a", "b", "mu", "sigma2")


@pytest.mark.parametrize("seed,kw", [(9000, {}), (9001, dict(n_pyr_levels=5)), (9002, dict(baseline=0.3)),
                                     (9003, dict(cam="QVGA")), (9004, dict(edgelet_frac=0.8))])
def test_oracle_seed_update_is_bit_identical_to_the_reference_tus(request, oracle, abi, synth, seed, kw):
    oracle.build_ref()
    kw = dict(kw)
    if "cam" in kw:
        kw["cam"] = getattr(synth, kw["cam"])
    d = synth.make_seed_batch(n=1200, seed=seed, **kw)
    o = oracle.seed_update(abi, d, 4)
    r = Reference(request.node.name, d, lambda: oracle.ref_seed_update(abi, d), SEED_FIELDS)
    alive = r.array("status") == 0  # the reference erases a seed whose variance reaches exactly 0 (converged): state not readable
    assert alive.mean() > 0.99
    for f in ("a", "b", "mu", "sigma2"):
        r.assert_equal(f, getattr(o, f)[alive], select=alive)
    assert set(np.unique(o.status)) == {0, 1, 2}


@pytest.mark.parametrize("opts", [dict(align_1d=True), dict(subpix_refinement=False), dict(edgelet_filtering=False),
                                  dict(max_epi_search_steps=40)])
def test_oracle_seed_update_matcher_options(request, oracle, abi, synth, opts):
    oracle.build_ref()
    d = synth.make_seed_batch(n=800, seed=9010)
    for k, v in opts.items():
        setattr(d, k, v)
    o = oracle.seed_update(abi, d, 4)
    r = Reference(request.node.name, d, lambda: oracle.ref_seed_update(abi, d), SEED_FIELDS)
    alive = r.array("status") == 0
    for f in ("a", "b", "mu", "sigma2"):
        r.assert_equal(f, getattr(o, f)[alive], select=alive)


def test_oracle_seed_update_measures_depth_and_shrinks_the_variance(oracle, abi, synth):
    d = synth.make_seed_batch(n=1500, seed=9020, edgelet_frac=0.0)
    o = oracle.seed_update(abi, d, 4)
    up = o.status == abi.SEED_UPDATED
    assert up.mean() > 0.7
    prior = np.abs(1.0 / d.mu[up] - d.depth_gt[up])
    meas = np.abs(o.depth[up] - d.depth_gt[up])
    assert np.median(meas) < 0.3 * np.median(prior)
    assert np.median(o.sigma2[up] / d.sigma2[up]) < 0.7
    nm = o.status == abi.SEED_NO_MATCH
    np.testing.assert_array_equal(o.b[nm], d.b[nm] + 1)
    nv = o.status == abi.SEED_NOT_VISIBLE
    np.testing.assert_array_equal(o.mu[nv], d.mu[nv])


@pytest.mark.gpu
@pytest.mark.parametrize("seed,kw", [(9100, {}), (9101, dict(n_pyr_levels=5, baseline=0.25)), (9102, dict(edgelet_frac=0.6))])
def test_gpu_seed_update_matches_the_oracle(pkg, oracle, abi, synth, gen_device, seed, kw):
    d = synth.make_seed_batch(n=6000, seed=seed, device=gen_device, **kw)
    ref = oracle.seed_update(abi, d, 8)
    out = pkg.DepthFilter().updatePointSeeds(d)
    # integer / exact part: which branch every seed took, the position found and the triangulated depth
    np.testing.assert_array_equal(out.status, ref.status)
    fin = np.isfinite(ref.px_cur).all(axis=1)
    np.testing.assert_array_equal(np.isfinite(out.px_cur).all(axis=1), fin)
    np.testing.assert_array_equal(out.px_cur[fin], ref.px_cur[fin])
    up = ref.status == abi.SEED_UPDATED
    np.testing.assert_array_equal(out.depth[up], ref.depth[up])
    assert np.isnan(out.depth[~up]).all()
    # untouched / b+1 seeds are exact; updated seeds agree to float round-off of the libm calls
    same = ~up
    for f in ("a", "b", "mu", "sigma2"):
        np.testing.assert_array_equal(getattr(out, f)[same], getattr(ref, f)[same], err_msg=f)
    ok = up & np.isfinite(ref.a) & np.isfinite(ref.sigma2)
    np.testing.assert_allclose(out.mu[ok], ref.mu[ok], rtol=2e-6, atol=0)
    # sigma2 = C1*(s2+m^2) + C2*(sigma2+mu^2) - mu_new^2 is a difference of O(mu^2) terms evaluated in float: its absolute
    # error is a few ulps of mu^2 (~3e-8 each) whatever the size of the result, hence the absolute tolerance
    np.testing.assert_allclose(out.sigma2[ok], ref.sigma2[ok], rtol=2e-4, atol=5e-7)
    # a and b come out of (e-f)/(f-e/f), a difference of nearly equal floats: round-off is amplified
    np.testing.assert_allclose(out.a[ok], ref.a[ok], rtol=5e-2)
    np.testing.assert_allclose(out.b[ok], ref.b[ok], rtol=5e-2, atol=1e-3)
    assert (out.converged == ref.converged).mean() > 0.999


@pytest.mark.gpu
def test_gpu_seed_update_options_and_bad_input(pkg, oracle, abi, synth, gen_device):
    import ctypes as C

    d = synth.make_seed_batch(n=1500, seed=9200, device=gen_device)
    for opts in (dict(align_1d=True), dict(subpix_refinement=False), dict(max_epi_search_steps=40)):
        for k, v in opts.items():
            setattr(d, k, v)
        ref = oracle.seed_update(abi, d, 8)
        out = pkg.DepthFilter().updatePointSeeds(d)
        np.testing.assert_array_equal(out.status, ref.status)
        up = ref.status == abi.SEED_UPDATED
        np.testing.assert_array_equal(out.depth[up], ref.depth[up])
    ctx = pkg.default_context()
    b, keep = abi.make_seed_batch(d)
    b.cur_pitch[1] = b.cur_pitch[1] + 16  # not dense
    out = abi.SeedOut(d.n)
    assert ctx.lib.plsvo_seed_update_batch_run(ctx.handle, C.byref(b), C.byref(out.struct)) == abi.ERR_INVALID


# ---- line seeds: DepthFilter::updateLineSeeds (src/depth_filter.cpp:367-471) -------------------------------------
LINE_FIELDS = ("a", "b", "mu", "sigma2", "mu_e", "sigma2_e")


@pytest.mark.parametrize("seed,kw", [(9500, {}), (9501, dict(n_pyr_levels=5)), (9502, dict(baseline=0.3)), (9503, dict(cam="QVGA"))])
def test_oracle_line_seed_update_is_bit_identical_to_the_reference_tus(request, oracle, abi, synth, seed, kw):
    oracle.build_ref()
    kw = dict(kw)
    if "cam" in kw:
        kw["cam"] = getattr(synth, kw["cam"])
    d = synth.make_line_seed_batch(n=1000, seed=seed, **kw)
    o = oracle.line_seed_update(abi, d, 4)
    r = Reference(request.node.name, d, lambda: oracle.ref_line_seed_update(abi, d), ("status",) + LINE_FIELDS)
    alive = r.array("status") == 0
    assert alive.mean() > 0.99
    for f in LINE_FIELDS:
        r.assert_equal(f, getattr(o, f)[alive], select=alive)
    assert set(np.unique(o.status)) == {0, 1, 2}
    for opts in (dict(align_1d=True), dict(subpix_refinement=False), dict(max_epi_search_steps=30)):
        for k, v in opts.items():
            setattr(d, k, v)
        o = oracle.line_seed_update(abi, d, 4)
        r = Reference(f"{request.node.name}/{opts}", d, lambda: oracle.ref_line_seed_update(abi, d), ("status",) + LINE_FIELDS)
        alive = r.array("status") == 0
        for f in LINE_FIELDS:
            r.assert_equal(f, getattr(o, f)[alive], select=alive, err_msg=f"{opts} {f}")


@pytest.mark.gpu
@pytest.mark.parametrize("seed,kw", [(9600, {}), (9601, dict(n_pyr_levels=5, baseline=0.25))])
def test_gpu_line_seed_update_matches_the_oracle(pkg, oracle, abi, synth, gen_device, seed, kw):
    d = synth.make_line_seed_batch(n=5000, seed=seed, device=gen_device, **kw)
    ref = oracle.line_seed_update(abi, d, 8)
    out = pkg.DepthFilter().updateLineSeeds(d)
    np.testing.assert_array_equal(out.status, ref.status)
    up = ref.status == abi.SEED_UPDATED
    np.testing.assert_array_equal(out.depth[up], ref.depth[up])      # z_s: exact
    np.testing.assert_array_equal(out.depth_e[up], ref.depth_e[up])  # z_e: exact
    assert np.isnan(out.depth[~up]).all() and np.isnan(out.depth_e[~up]).all()
    for f in ("px_cur", "px_cur_e"):  # Matcher::px_cur_ after the start / end search: exact, NaN in the same places
        o, r = getattr(out, f), getattr(ref, f)
        fin = np.isfinite(r).all(axis=1)
        np.testing.assert_array_equal(np.isfinite(o).all(axis=1), fin, err_msg=f)
        np.testing.assert_array_equal(o[fin], r[fin], err_msg=f)
    assert np.isfinite(ref.px_cur_e[up]).all()
    for f in LINE_FIELDS:
        np.testing.assert_array_equal(getattr(out, f)[~up], getattr(ref, f)[~up], err_msg=f)
    ok = up & np.isfinite(ref.a) & np.isfinite(ref.sigma2) & np.isfinite(ref.sigma2_e)
    for f in ("mu", "mu_e"):
        np.testing.assert_allclose(getattr(out, f)[ok], getattr(ref, f)[ok], rtol=2e-6, atol=0, err_msg=f)
    for f in ("sigma2", "sigma2_e"):
        np.testing.assert_allclose(getattr(out, f)[ok], getattr(ref, f)[ok], rtol=2e-4, atol=5e-7, err_msg=f)
    np.testing.assert_allclose(out.a[ok], ref.a[ok], rtol=5e-2)
    np.testing.assert_allclose(out.b[ok], ref.b[ok], rtol=5e-2, atol=1e-3)
    assert (out.converged == ref.converged).mean() > 0.999
