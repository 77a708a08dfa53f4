"""feature_alignment::align2D (src/feature_alignment.cpp:160-290), SURVEY §8f rank 1.
fp32 sequential arithmetic: the GPU kernel (thread per feature) must be bit-identical to the oracle."""
import numpy as np
import pytest
import torch

from reference_outputs import Reference


def _case(synth, n=400, seed=7, device="cpu"):
    rng = np.random.default_rng(seed)
    cam = synth.VGA
    scene = synth.Scene()
    poses = synth.pose7_from_Rt(*synth.se3_exp_Rt(torch.tensor(rng.uniform(-0.05, 0.05, (3, 6)), dtype=torch.float64)))
    img0 = scene.render(cam, poses.to(device)).cpu()
    pyr = {l: np.ascontiguousarray(p.numpy()) for l, p in enumerate(synth.build_pyramid(img0, 3))}
    image_index = rng.integers(0, 3, n).astype(np.int32)
    level = rng.integers(0, 3, n).astype(np.int32)
    border = np.zeros((n, 10, 10), np.uint8)
    truth = np.zeros((n, 2))
    for i in range(n):
        im = pyr[int(level[i])][int(image_index[i])]
        h, w = im.shape
        xi, yi = rng.integers(12, w - 12), rng.integers(12, h - 12)
        border[i] = im[yi - 5:yi + 5, xi - 5:xi + 5]
        truth[i] = (xi, yi)
    ref = np.ascontiguousarray(border[:, 1:9, 1:9])
    px0 = truth + rng.uniform(-1.5, 1.5, (n, 2))
    # a few features start outside the frame / on the border: the loop must break without converging
    px0[:5] = [[1.0, 1.0], [2.5, 100.0], [-3.0, 5.0], [1e6, 10.0], [float("nan"), 3.0]]
    return cam, pyr, image_index, level, border, ref, px0, truth


def test_oracle_align2d_converges_to_the_true_position(oracle, abi, synth):
    cam, pyr, idx, lvl, border, ref, px0, truth = _case(synth, n=200)
    conv, px = oracle.align2d(abi, pyr, idx, lvl, border, ref, px0, 10)
    assert not conv[:5].any()
    ok = conv[5:]
    assert ok.mean() > 0.9
    err = np.abs(px[5:] - truth[5:]).max(axis=1)
    assert np.median(err[ok]) < 0.02 and (err[ok] < 0.2).mean() > 0.97


@pytest.mark.gpu
def test_gpu_align2d_is_bit_identical_to_the_oracle(pkg, oracle, abi, synth, gen_device):
    cam, pyr, idx, lvl, border, ref, px0, truth = _case(synth, n=2000, seed=8, device=gen_device)
    conv_ref, px_ref = oracle.align2d(abi, pyr, idx, lvl, border, ref, px0, 10)
    conv, px = pkg.feature_alignment.align2D(pyr, idx, lvl, border, ref, 10, px0, cam.width, cam.height)
    np.testing.assert_array_equal(conv, conv_ref)
    finite = np.isfinite(px_ref).all(axis=1)
    np.testing.assert_array_equal(px[finite], px_ref[finite])
    assert (np.isnan(px[~finite]) == np.isnan(px_ref[~finite])).all()


def test_oracle_align2d_is_bit_identical_to_the_reference_tu(request, oracle, abi, synth):
    """oracle/_ref compiles the reference's own src/feature_alignment.cpp in place (oracle/ref_harness.cpp);
    the restatement must reproduce align2D's converged flags and refined positions bit for bit."""
    oracle.build_ref()
    for seed, n_iter in ((9, 10), (10, 3), (11, 30)):
        cam, pyr, idx, lvl, border, ref, px0, truth = _case(synth, n=600, seed=seed)
        conv_o, px_o = oracle.align2d(abi, pyr, idx, lvl, border, ref, px0, n_iter)
        r = Reference(f"{request.node.name}/{seed}", (pyr, idx, lvl, border, ref, px0, n_iter), lambda: dict(zip(
            ("conv", "px"), oracle.ref_align2d(abi, pyr, idx, lvl, border, ref, px0, n_iter))))
        r.assert_equal("conv", conv_o)
        r.assert_equal("px", px_o)  # NaN == NaN under assert_array_equal


# ---- align1D (src/feature_alignment.cpp:40-157): 1 DoF along a direction -----------------------------
def _dirs(n, seed):
    rng = np.random.default_rng(seed)
    ang = rng.uniform(0, 2 * np.pi, n)
    d = np.stack([np.cos(ang), np.sin(ang)], -1).astype(np.float32)
    d[:3] = [[1, 0], [0, 1], [0.6, 0.8]]
    return d


def test_oracle_align1d_is_bit_identical_to_the_reference_tu(request, oracle, abi, synth):
    oracle.build_ref()
    for seed, n_iter in ((19, 10), (20, 3), (21, 30)):
        cam, pyr, idx, lvl, border, ref, px0, truth = _case(synth, n=600, seed=seed)
        d = _dirs(600, seed)
        conv_o, px_o, h_o = oracle.align1d(abi, pyr, idx, lvl, d, border, ref, px0, n_iter)
        r = Reference(f"{request.node.name}/{seed}", (pyr, idx, lvl, d, border, ref, px0, n_iter), lambda: dict(zip(
            ("conv", "px", "h_inv"), oracle.ref_align1d(abi, pyr, idx, lvl, d, border, ref, px0, n_iter))))
        r.assert_equal("conv", conv_o)
        r.assert_equal("px", px_o)
        r.assert_equal("h_inv", h_o)
        assert conv_o[5:].mean() > 0.3  # 1-DoF search converges when the offset has a component along dir


@pytest.mark.gpu
def test_gpu_align1d_is_bit_identical_to_the_oracle(pkg, oracle, abi, synth, gen_device):
    cam, pyr, idx, lvl, border, ref, px0, truth = _case(synth, n=2000, seed=22, device=gen_device)
    d = _dirs(2000, 22)
    conv_ref, px_ref, h_ref = oracle.align1d(abi, pyr, idx, lvl, d, border, ref, px0, 10)
    conv, px, h = pkg.feature_alignment.align1D(pyr, idx, lvl, d, border, ref, 10, px0, cam.width, cam.height)
    np.testing.assert_array_equal(conv, conv_ref)
    np.testing.assert_array_equal(h, h_ref)
    finite = np.isfinite(px_ref).all(axis=1)
    np.testing.assert_array_equal(px[finite], px_ref[finite])
    assert (np.isnan(px[~finite]) == np.isnan(px_ref[~finite])).all()
