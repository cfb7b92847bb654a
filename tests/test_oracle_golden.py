"""Pin the oracle: replay the reference's own outputs (tests/golden, made by oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

import rgbd_b200  # noqa: F401
from rgbd_b200 import synthetic
from oracle import hotpath as O
from oracle import weights as OW
from oracle.make_golden import decompose_cases, load_wiring


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_decompose_bit_exact(golden_dir):
    g = _load(golden_dir, "decompose.npz")
    cases = decompose_cases(synthetic)
    assert [c[0] for c in cases] == list(g["names"])
    seen_nmasks = set()
    for name, gray, ratio in cases:
        dec = O.depth_decompose(gray, ratio)
        np.testing.assert_array_equal(dec["hist"], g[f"{name}.hist"], err_msg=name)
        np.testing.assert_array_equal(dec["edges"], g[f"{name}.edges"], err_msg=name)
        np.testing.assert_array_equal(np.array(dec["centres"], dtype=np.float32), g[f"{name}.modes"], err_msg=name)
        wins = np.array([[a, b] for a, b in dec["windows"]], dtype=np.float32).reshape(-1, 2)
        np.testing.assert_array_equal(wins, g[f"{name}.windows"], err_msg=name)
        packed = np.packbits(np.stack(dec["masks"]).astype(np.uint8), axis=None)
        assert len(dec["masks"]) == int(g[f"{name}.nmasks"]), name
        np.testing.assert_array_equal(packed, g[f"{name}.masks"], err_msg=name)
        seen_nmasks.add((len(dec["centres"]), len(dec["masks"])))
    # the fixture set covers 0, <3 and 3 surviving modes (SURVEY H4)
    assert any(m == 0 for m, _ in seen_nmasks) and any(m == 3 for m, _ in seen_nmasks)
    assert any(0 < m < 3 for m, _ in seen_nmasks)


def test_histogram_matches_numpy_directly():
    rs = np.random.RandomState(3)
    for trial in range(60):
        n = rs.randint(10, 5000)
        lo, hi = np.sort(rs.randn(2) * 10 ** rs.uniform(-3, 3))
        a = rs.uniform(lo, hi, size=n).astype(np.float32)
        if trial % 5 == 0:
            a = np.round(a, 1)
        hist, edges = O.depth_histogram(a)
        rh, re = np.histogram(a, bins=512, range=(np.nanmin(a), np.nanmax(a)))
        np.testing.assert_array_equal(hist, rh)
        np.testing.assert_array_equal(edges, re)


def test_peaks_match_scipy_directly():
    from scipy.signal import find_peaks
    rs = np.random.RandomState(4)
    for trial in range(300):
        kind = trial % 4
        if kind == 0:
            h = rs.randint(0, 50, size=512)
        elif kind == 1:
            h = np.repeat(rs.randint(0, 9, size=64), 8)            # plateaus
        elif kind == 2:
            h = np.zeros(512, dtype=np.int64)
            h[rs.randint(0, 512, size=12)] = rs.randint(1, 1000, size=12)   # sparse
        else:
            x = np.arange(512)
            h = sum((rs.randint(100, 3000) * np.exp(-0.5 * ((x - rs.randint(0, 512)) / rs.uniform(2, 30)) ** 2))
                    for _ in range(4)).astype(np.int64) + rs.randint(0, 5, size=512)
        h = h.astype(np.int64)
        ref, _ = find_peaks(h, prominence=0.01 * np.max(h))
        peaks = O.local_maxima_1d(list(h))
        proms = O.peak_prominences(list(h), peaks)
        kept = [p for p, pr in zip(peaks, proms) if 0.01 * float(h.max()) <= float(pr)]
        assert kept == list(ref)


def test_gray(golden_dir):
    g = _load(golden_dir, "gray.npz")["gray"]
    d3 = (np.random.RandomState(11).randn(3, 40, 56) * 1.3).astype(np.float32)
    np.testing.assert_array_equal(O.to_grayscale(d3)[None], g)


def _gray_for(j, kind, dhw):
    _, d = synthetic.synth_rgbd_u8(20 + j, dhw[0], dhw[1], kind)
    return O.to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))


@pytest.mark.parametrize("tag,ci,co,hw,dhw", [("proj", 8, 16, (24, 32), (96, 128)),
                                              ("ident", 8, 8, (24, 32), (96, 128)),
                                              ("proj_odd", 8, 24, (15, 20), (60, 80))])
def test_dsam_forward(golden_dir, tag, ci, co, hw, dhw):
    g = _load(golden_dir, "dsam.npz")
    w = OW.dsam_weights(ci, co, seed=100 + ci + co)
    feat = torch.from_numpy(np.random.RandomState(5).randn(1, ci, *hw).astype(np.float32))
    for j, kind in enumerate(["nyu", "constant", "two_valued"]):
        y = O.dsam_forward(w, feat, _gray_for(j, kind, dhw), 0.3)
        ref = g[f"{tag}.{kind}"]
        assert y.shape == ref.shape
        np.testing.assert_allclose(y.numpy(), ref, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("tag,hw,sizes", [("even", (64, 96), [(16, 24), (8, 12), (4, 6), (2, 3)]),
                                          ("ragged", (50, 70), [(13, 18), (7, 9), (4, 5), (2, 3)])])
def test_dggm_forward(golden_dir, tag, hw, sizes):
    g = _load(golden_dir, "dggm.npz")
    chans = [4, 8, 12, 16]
    w = OW.dggm_weights(chans, 3, seed=300)
    rs = np.random.RandomState(9)
    feats = [torch.from_numpy(rs.randn(2, c, h, ww).astype(np.float32)) for c, (h, ww) in zip(chans, sizes)]
    grad = torch.from_numpy(rs.rand(2, 3, *hw).astype(np.float32))
    mask = torch.from_numpy((rs.rand(2, 1, *hw) < 0.6).astype(np.float32))
    ys = O.dggm_forward(w, feats, grad, mask)
    for i, y in enumerate(ys):
        np.testing.assert_allclose(y.numpy(), g[f"{tag}.{i}"], rtol=1e-5, atol=2e-6)
    # None gradient / mask -> passthrough (CM:1263-1265)
    ys = O.dggm_forward(w, feats, None, mask)
    assert all(a is b for a, b in zip(ys, feats))


def test_gradient_features_bit_exact(golden_dir):
    g = _load(golden_dir, "gradfeat.npz")
    for j, kind in enumerate(["nyu", "nyu", "constant", "two_valued", "all_invalid", "uniform"]):
        _, d = synthetic.synth_rgbd_u8(40 + j, 60, 84, kind)
        norm, gx, gy, vm = O.gradient_features(d)
        for name, arr in (("norm", norm), ("gx", gx), ("gy", gy), ("vmask", vm)):
            np.testing.assert_array_equal(arr, g[f"{kind}{j}.{name}"], err_msg=f"{kind}{j}.{name}")


def test_ratio_predictor(golden_dir):
    ref = _load(golden_dir, "ratio.npz")["ratio"]
    frames = []
    for j in range(2):
        _, d = synthetic.synth_rgbd_u8(60 + j, 48, 64, "nyu")
        frames.append(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
    r = O.ratio_predictor_forward(OW.ratio_weights(seed=500), torch.from_numpy(np.stack(frames)))
    np.testing.assert_allclose(r.numpy(), ref, rtol=1e-5, atol=1e-6)
    assert ((r >= 0.01) & (r <= 0.5)).all()


def test_wiring(golden_dir):
    g = load_wiring(golden_dir, "wiring.npz")
    w = OW.guidance_weights(seed=700)
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs))
    feats = [torch.from_numpy(g[f"feat{i}"]) for i in range(4)]
    fused, ratios = O.depth_guidance_forward(w, pv, feats)
    np.testing.assert_allclose(ratios.numpy(), g["ratios"], rtol=1e-5, atol=1e-6)
    for i in range(4):
        ref = g[f"fused{i}"]
        np.testing.assert_allclose(fused[i].numpy(), ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())


@pytest.mark.parametrize("version", ["0.0.3", "0.1.2"])
def test_other_version_wiring(golden_dir, version):
    g = load_wiring(golden_dir, f"wiring_v{version.replace('.', '')}.npz")
    w = OW.guidance_weights(seed=700)
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs))
    pvv = torch.cat([pv[:, 0:3], pv[:, 6:9], pv[:, 9:10]], dim=1) if version == "0.0.3" else pv[:, 0:6]
    feats = [torch.from_numpy(g[f"feat{i}"]) for i in range(4)]
    fused = O.version_forward(version, w, pvv, feats)
    for i in range(4):
        ref = g[f"fused{i}"]
        np.testing.assert_allclose(fused[i].numpy(), ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())


@pytest.mark.parametrize("version", ["0.1.3", "0.3.0"])
def test_depth_encoder_version_wiring(golden_dir, version):
    """CM:258-322: feature-based RatioPredictor -> DSAM cascade (-> DGGM on the result for 0.3.0), reference goldens."""
    g = load_wiring(golden_dir, f"wiring_v{version.replace('.', '')}.npz")
    w = OW.guidance_weights_feature_ratio(seed=700)
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs))
    feats = [torch.from_numpy(g[f"feat{i}"]) for i in range(4)]
    dfeats = [torch.from_numpy(g[f"dfeat{i}"]) for i in range(4)]
    ratios = O.ratio_from_features_forward({k[len("ratio_predictor."):]: v for k, v in w.items()
                                            if k.startswith("ratio_predictor.")}, dfeats)
    np.testing.assert_allclose(ratios.numpy(), g["ratios"], rtol=1e-5)
    fused = O.version_forward(version, w, pv, feats, dfeats)
    for i in range(4):
        ref = g[f"fused{i}"]
        np.testing.assert_allclose(fused[i].numpy(), ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())


def test_front_end_matches_huggingface_processor_and_reference_mapper(golden_dir):
    """DL:386-425: pixel_values of map_10channel_case2 from the real HF (PIL backend) processor with the reference's
    preprocessor_config.json + the reference's calculate_gradient_features, against the restatement the synthetic input
    builder and the device front-end share (bit-exact, including the checkpoint's one-ulp-low std[1])."""
    g = _load(golden_dir, "frontend.npz")
    assert np.array_equal(g["image_mean"].astype(np.float32), synthetic.IMAGE_MEAN)
    assert np.array_equal(g["image_std"].astype(np.float32), synthetic.IMAGE_STD)
    assert float(g["rescale_factor"]) == synthetic.RESCALE_FACTOR
    for j in range(3):
        pv = synthetic.assemble_pixel_values(g[f"f{j}.rgb"], g[f"f{j}.depth"], O.gradient_features)
        assert pv.dtype == np.float32 and np.array_equal(pv, g[f"f{j}.pixel_values"])


def test_ratio_predictor_train_mode_matches_reference_golden(golden_dir):
    """oracle.ratio_predictor_forward_train == the reference module in .train() (batch-statistics BatchNorm, running
    statistics after each of two steps, injected Dropout keep-masks); golden from oracle/make_golden_train.py."""
    from oracle.make_golden_train import SEED_W, train_inputs
    g = np.load(os.path.join(golden_dir, "ratio_train.npz"))
    w = OW.ratio_weights(seed=SEED_W)
    for step in range(2):
        x, keep = train_inputs(synthetic, step)
        r, w = O.ratio_predictor_forward_train(w, x, keep)
        np.testing.assert_allclose(r.numpy(), g[f"step{step}.ratio"], rtol=1e-5, atol=1e-7)
        for k in w:
            if "running" in k:
                np.testing.assert_allclose(w[k].numpy(), g[f"step{step}.{k}"], rtol=2e-5, atol=1e-6, err_msg=k)
            elif "num_batches" in k:
                assert int(w[k]) == int(g[f"step{step}.{k}"]) == step + 1
