"""Golden vector of the v0.4.0 wiring (CM:324-355) at the benchmarked size -> tests/golden/wiring_480x640.npz.

    python oracle/make_golden_fullsize.py

One synthetic 480x640 frame, the guidance weights of seed 700 and seeded Swin-T-shaped encoder features (the features are
regenerated from the seed, not stored).  Stored: the predicted ratio, the SHA-256 and per-channel sums of the pixel values
(gradient features included), and for each of the four fused maps the channel means, the largest magnitude and a fixed sample
of its elements with their flat indices.

The values come from the port (oracle.hotpath).  tests/test_oracle_vs_reference.py compares the port with the reference
itself at this size wherever the reference project is importable (max relative difference of the fused maps 0 / 0 / 4e-8 /
2e-8 when it was run), and with this file everywhere.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.make_golden import GOLD, load_pkg      # noqa: E402

H, W = 480, 640
CHANNELS = (96, 192, 384, 768)
STRIDES = (4, 8, 16, 32)
SAMPLE = 16384                 # elements kept per fused map


def fullsize_inputs(synthetic, gradient_features):
    """(pixel_values (1,10,H,W), encoder features) of the stored case."""
    rgb, d = synthetic.synth_rgbd_u8(1234, H, W, "nyu")
    pv = torch.from_numpy(synthetic.assemble_pixel_values(rgb, d, gradient_features))[None]
    g = torch.Generator().manual_seed(4800)
    feats = [torch.randn(1, c, H // s, W // s, generator=g) for c, s in zip(CHANNELS, STRIDES)]
    return pv, feats


def pixel_values_digest(pv: torch.Tensor) -> str:
    return hashlib.sha256(np.ascontiguousarray(pv.numpy()).tobytes()).hexdigest()


def main():
    from oracle import hotpath as O
    synthetic, weights = load_pkg()
    pv, feats = fullsize_inputs(synthetic, O.gradient_features)
    with torch.no_grad():
        fused, ratios = O.depth_guidance_forward(weights.guidance_weights(seed=700), pv, feats)
    out = {"ratios": ratios.numpy(), "pixel_values.sha256": np.array(pixel_values_digest(pv)),
           "pixel_values.channel_sums": pv.double().sum(dim=(0, 2, 3)).numpy()}
    for i, f in enumerate(fused):
        flat = f.reshape(-1).numpy()
        idx = np.sort(np.random.default_rng(i).choice(flat.size, SAMPLE, replace=False))
        out[f"fused{i}.index"] = idx.astype(np.int64)
        out[f"fused{i}.sample"] = flat[idx]
        out[f"fused{i}.channel_mean"] = f.double().mean(dim=(0, 2, 3)).numpy()
        out[f"fused{i}.absmax"] = np.array(float(f.abs().max()))
    path = os.path.join(GOLD, "wiring_480x640.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), out["ratios"].ravel())


if __name__ == "__main__":
    main()
