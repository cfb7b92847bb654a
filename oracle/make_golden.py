"""Generate tests/golden/*.npz from the REFERENCE ITSELF (run in the build container only).

    python oracle/make_golden.py            # needs /root/reference (read-only)

The reference is imported unmodified with the two import shims of SURVEY.md §8c (a stub
``matplotlib`` and the relocated ``load_backbone``).  Inputs and weights are regenerated in
the tests from frozen ``RandomState`` seeds (oracle/weights.py, synthetic.py); only the
reference's OUTPUTS (and inputs that cannot be regenerated, e.g. Swin features) are stored.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
GOLD = os.path.join(ROOT, "tests", "golden")
# Every wiring golden is computed from the same colour-encoder features (one seed, one config) and both depth-encoder versions
# from the same depth-encoder features: each set is stored once, beside the per-version outputs, so no file grows past 1 MB.
WIRING_INPUTS = {"feat": "wiring_feat.npz", "dfeat": "wiring_dfeat.npz"}


def save_wiring(name, out, gold=GOLD):
    """Write the wiring golden ``name`` (``fused*``, ``ratios``) and the encoder features (``feat*``, ``dfeat*``) in ``out``.
    Features already stored by another wiring golden must be equal to the ones given here: the other goldens' outputs were
    computed from them."""
    out = dict(out)
    for prefix, shared in WIRING_INPUTS.items():
        feats = {k: out.pop(k) for k in [k for k in out if k.rstrip("0123456789") == prefix]}
        if not feats:
            continue
        path = os.path.join(gold, shared)
        if os.path.exists(path):
            old = np.load(path)
            if sorted(old.files) != sorted(feats) or not all(np.array_equal(old[k], v) for k, v in feats.items()):
                raise ValueError(f"{name}: its {prefix}* differ from those in {shared}, which other wiring goldens were made "
                                 f"from; remove {shared} and regenerate every wiring golden")
        else:
            np.savez_compressed(path, **feats)
    np.savez_compressed(os.path.join(gold, name), **out)


def load_wiring(gold, name):
    """The wiring golden ``name`` together with the encoder features it was computed from (``feat*``, ``dfeat*``)."""
    g = dict(np.load(os.path.join(gold, name)))
    for shared in WIRING_INPUTS.values():
        g.update(np.load(os.path.join(gold, shared)))
    return g


def import_reference():
    for name in ("matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    import transformers.backbone_utils as bu
    import transformers.utils.backbone_utils as old
    if not hasattr(old, "load_backbone"):
        old.load_backbone = bu.load_backbone
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import mask2former.utils.custom_model as cm
    import mask2former.utils.data_process as dp
    return cm, dp


def load_pkg():
    sys.path.insert(0, ROOT)
    import rgbd_b200  # noqa: F401  (root shim for the hyphenated package directory)
    from rgbd_b200 import synthetic
    from oracle import weights
    return synthetic, weights


def decompose_cases(synthetic):
    """(name, gray float32 (H,W), ratio) cases for the integer path, incl. SURVEY §8c edge cases."""
    from oracle.hotpath import to_grayscale
    cases = []
    H, W = 96, 128
    for i, kind in enumerate(["nyu", "nyu", "nyu", "uniform", "constant", "two_valued", "all_invalid"]):
        _, d = synthetic.synth_rgbd_u8(i, H, W, kind)
        d3 = synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2))
        cases.append((f"{kind}{i}", to_grayscale(d3), [0.01, 0.1, 0.37, 0.5][i % 4]))
    rs = np.random.RandomState(7)
    g = (rs.rand(64, 64) * 5.0).astype(np.float32)          # exp6_dsam.py:37-60 smoke input
    g[10:20, 10:20] += 2.0
    g[40:50, 40:50] += 4.0
    g[g < 0.5] = np.nan
    cases.append(("exp6_nan", g, 0.1))
    g2 = (rs.randn(80, 112) * 0.3).astype(np.float32)        # negative mode centres -> empty masks
    g2[:40] -= 1.5
    g2[40:] += 0.8
    cases.append(("negative_centres", g2, 0.3))
    g3 = np.round(rs.rand(72, 96) * 20).astype(np.float32) / 4  # plateaus / ties in the histogram
    cases.append(("quantised", g3, 0.25))
    g4 = np.concatenate([np.full(3000, 1.0), np.full(3000, 2.0), np.full(3000, 3.0), np.full(288, 0.0),
                         np.full(3000, 4.0)]).astype(np.float32).reshape(96, -1)
    cases.append(("tied_heights", g4, 0.2))
    return cases


def main():
    torch.manual_seed(0)
    cm, dp = import_reference()
    synthetic, weights = load_pkg()
    os.makedirs(GOLD, exist_ok=True)

    # ---- 1. integer path: histogram / modes / windows / masks -------------------------------
    dsam = cm.DSAModule(8, 16, 3)
    out = {}
    names = []
    for name, gray, ratio in decompose_cases(synthetic):
        names.append(name)
        hist, edges = dsam._calculate_depth_histogram(gray)
        modes = dsam._select_depth_distribution_modes(hist, edges, num_modes=3)
        out[f"{name}.hist"] = hist.astype(np.int64)
        out[f"{name}.edges"] = edges.astype(np.float32)
        out[f"{name}.modes"] = np.array(modes, dtype=np.float32)
        if modes:
            wins = dsam._define_depth_interval_windows(modes, window_size_ratio=ratio)
            masks = dsam._generate_depth_region_masks(gray, wins)
            out[f"{name}.windows"] = np.array([[float(a), float(b)] for a, b in wins], dtype=np.float32)
        else:
            masks = [np.zeros_like(gray, dtype=bool)] * 4
            out[f"{name}.windows"] = np.zeros((0, 2), dtype=np.float32)
        out[f"{name}.masks"] = np.packbits(np.stack(masks).astype(np.uint8), axis=None)
        out[f"{name}.nmasks"] = np.array(len(masks))
    out["names"] = np.array(names)
    np.savez_compressed(os.path.join(GOLD, "decompose.npz"), **out)

    # ---- 2. to_grayscale ---------------------------------------------------------------------
    plm = cm.CustomMask2FormerPixelLevelModule.__new__(cm.CustomMask2FormerPixelLevelModule)
    rs = np.random.RandomState(11)
    d3 = (rs.randn(3, 40, 56) * 1.3).astype(np.float32)
    g = cm.CustomMask2FormerPixelLevelModule.to_grayscale(plm, torch.from_numpy(d3))
    np.savez_compressed(os.path.join(GOLD, "gray.npz"), gray=g.numpy())

    # ---- 3. DSAModule forward (projection and identity variants) ----------------------------
    out = {}
    for tag, (ci, co), hw, dhw in (("proj", (8, 16), (24, 32), (96, 128)), ("ident", (8, 8), (24, 32), (96, 128)),
                                   ("proj_odd", (8, 24), (15, 20), (60, 80))):
        m = cm.DSAModule(ci, co, 3)
        w = weights.dsam_weights(ci, co, seed=100 + ci + co)
        m.load_state_dict(w)
        m.eval()
        rs = np.random.RandomState(5)
        feat = torch.from_numpy(rs.randn(1, ci, *hw).astype(np.float32))
        for j, kind in enumerate(["nyu", "constant", "two_valued"]):
            from oracle.hotpath import to_grayscale
            _, d = synthetic.synth_rgbd_u8(20 + j, dhw[0], dhw[1], kind)
            gray = to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
            with torch.no_grad():
                y = m(feat, torch.from_numpy(gray)[None], 0.3)
            out[f"{tag}.{kind}"] = y.numpy()
    np.savez_compressed(os.path.join(GOLD, "dsam.npz"), **out)

    # ---- 4. DGGM forward ------------------------------------------------------------------------
    out = {}
    for tag, chans, (H, W), sizes in (
            ("even", [4, 8, 12, 16], (64, 96), [(16, 24), (8, 12), (4, 6), (2, 3)]),
            ("ragged", [4, 8, 12, 16], (50, 70), [(13, 18), (7, 9), (4, 5), (2, 3)])):
        m = cm.DepthGradientInjectionResidual(chans, 3)
        m.load_state_dict(weights.dggm_weights(chans, 3, seed=300))
        rs = np.random.RandomState(9)
        feats = [torch.from_numpy(rs.randn(2, c, h, w).astype(np.float32)) for c, (h, w) in zip(chans, sizes)]
        grad = torch.from_numpy(rs.rand(2, 3, H, W).astype(np.float32))
        mask = torch.from_numpy((rs.rand(2, 1, H, W) < 0.6).astype(np.float32))
        with torch.no_grad():
            ys = m(feats, grad, mask)
        for i, y in enumerate(ys):
            out[f"{tag}.{i}"] = y.numpy()
    np.savez_compressed(os.path.join(GOLD, "dggm.npz"), **out)

    # ---- 5. gradient features (offline half of DGGM) ---------------------------------------------
    out = {}
    for j, kind in enumerate(["nyu", "nyu", "constant", "two_valued", "all_invalid", "uniform"]):
        _, d = synthetic.synth_rgbd_u8(40 + j, 60, 84, kind)
        norm, gx, gy, vm = dp.calculate_gradient_features(d)
        out[f"{kind}{j}.norm"] = norm
        out[f"{kind}{j}.vmask"] = vm
        out[f"{kind}{j}.gx"] = gx
        out[f"{kind}{j}.gy"] = gy
    np.savez_compressed(os.path.join(GOLD, "gradfeat.npz"), **out)

    # ---- 6. ratio predictor (eval) -----------------------------------------------------------------
    m = cm.EnhancedDepthImageRatioPredictor(3)
    m.load_state_dict(weights.ratio_weights(seed=500))
    m.eval()
    frames = []
    for j in range(2):
        _, d = synthetic.synth_rgbd_u8(60 + j, 48, 64, "nyu")
        frames.append(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
    with torch.no_grad():
        r = m(torch.from_numpy(np.stack(frames)))
    np.savez_compressed(os.path.join(GOLD, "ratio.npz"), ratio=r.numpy())

    # ---- 7. v0.4.0 wiring: encoder features -> list handed to the pixel decoder (CM:324-355) ------
    cfg = cm.CustomConfig.from_pretrained(os.path.join(REF, "mask2former/checkpoints/standard"))
    torch.manual_seed(42)
    plm = cm.CustomMask2FormerPixelLevelModule(cfg, version="0.4.0")
    w = weights.guidance_weights(seed=700)
    missing = plm.load_state_dict(w, strict=False)
    assert not missing.unexpected_keys, missing.unexpected_keys
    plm.eval()
    from oracle.hotpath import gradient_features
    H, W = 64, 96
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, H, W, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, lambda x: dp.calculate_gradient_features(x)))
    pv = torch.from_numpy(np.stack(pvs))
    captured = {}
    plm.encoder.register_forward_hook(lambda mod, a, o: captured.__setitem__("feats", [t.detach().clone() for t in o.feature_maps]))
    plm.decoder.register_forward_pre_hook(lambda mod, a: captured.__setitem__("fused", [t.detach().clone() for t in a[0]]))
    plm.ratio_predictor.register_forward_hook(lambda mod, a, o: captured.__setitem__("ratios", o.detach().clone()))
    with torch.no_grad():
        plm(pv)
    out = {"ratios": captured["ratios"].numpy()}
    for i in range(4):
        out[f"feat{i}"] = captured["feats"][i].numpy()
        out[f"fused{i}"] = captured["fused"][i].numpy()
    save_wiring("wiring.npz", out)
    # ---- 8. other version branches that reuse DGGM / DSAM (CM:156-163, CM:234-256) ---------------------------
    for version, nch in (("0.0.3", 7), ("0.1.2", 6)):
        torch.manual_seed(42)
        plm = cm.CustomMask2FormerPixelLevelModule(cfg, version=version)
        missing = plm.load_state_dict({k: v for k, v in w.items() if k.split(".")[0] in dict(plm.named_children())}, strict=False)
        assert not missing.unexpected_keys, missing.unexpected_keys
        plm.eval()
        if version == "0.0.3":      # rgb, gradient map (3 ch), gradient mask
            pvv = torch.cat([pv[:, 0:3], pv[:, 6:9], pv[:, 9:10]], dim=1)
        else:                        # rgb, depth
            pvv = pv[:, 0:6].clone()
        cap = {}
        plm.encoder.register_forward_hook(lambda mod, a, o: cap.__setitem__("feats", [t.detach().clone() for t in o.feature_maps]))
        plm.decoder.register_forward_pre_hook(lambda mod, a: cap.__setitem__("fused", [t.detach().clone() for t in a[0]]))
        with torch.no_grad():
            plm(pvv)
        out = {}
        for i in range(4):
            out[f"feat{i}"] = cap["feats"][i].numpy()
            out[f"fused{i}"] = cap["fused"][i].numpy()
        save_wiring(f"wiring_v{version.replace('.', '')}.npz", out)
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == "__main__":
    main()
