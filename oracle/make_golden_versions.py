"""Golden vectors of the version 0.1.3 / 0.3.0 branches (CM:258-322) from the REFERENCE module itself ->
tests/golden/wiring_v013.npz, wiring_v030.npz: predicted ratios and the list handed to the pixel decoder; the colour- and
depth-encoder features go to the shared wiring_feat.npz / wiring_dfeat.npz.  Run where the reference project is importable:
``python oracle/make_golden_versions.py``."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.make_golden import GOLD, REF, import_reference, load_pkg, save_wiring      # noqa: E402


def main():
    cm, dp = import_reference()
    synthetic, weights = load_pkg()
    cfg = cm.CustomConfig.from_pretrained(os.path.join(REF, "mask2former/checkpoints/standard"))
    w = weights.guidance_weights_feature_ratio(seed=700)
    H, W = 64, 96
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, H, W, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, lambda x: dp.calculate_gradient_features(x)))
    pv = torch.from_numpy(np.stack(pvs))
    for version in ("0.1.3", "0.3.0"):
        torch.manual_seed(42)
        plm = cm.CustomMask2FormerPixelLevelModule(cfg, version=version)
        own = dict(plm.named_children())
        missing = plm.load_state_dict({k: v for k, v in w.items() if k.split(".")[0] in own}, strict=False)
        assert not missing.unexpected_keys, missing.unexpected_keys
        plm.eval()
        pvv = pv[:, 0:6].clone() if version == "0.1.3" else pv.clone()
        cap = {}
        # the reference adds the DSAM outputs IN PLACE into the encoder's feature maps (CM:275): clone inside the hook
        plm.encoder.register_forward_hook(lambda mod, a, o: cap.__setitem__("feats", [t.detach().clone() for t in o.feature_maps]))
        plm.depth_encoder.register_forward_hook(lambda mod, a, o: cap.__setitem__("dfeats", [t.detach().clone() for t in o.feature_maps]))
        plm.ratio_predictor.register_forward_hook(lambda mod, a, o: cap.__setitem__("ratios", o.detach().clone()))
        plm.decoder.register_forward_pre_hook(lambda mod, a: cap.__setitem__("fused", [t.detach().clone() for t in a[0]]))
        with torch.no_grad():
            plm(pvv)
        out = {"ratios": cap["ratios"].numpy()}
        for i in range(4):
            out[f"feat{i}"] = cap["feats"][i].numpy()
            out[f"dfeat{i}"] = cap["dfeats"][i].numpy()
            out[f"fused{i}"] = cap["fused"][i].numpy()
        path = os.path.join(GOLD, f"wiring_v{version.replace('.', '')}.npz")
        save_wiring(os.path.basename(path), out)
        print(path, os.path.getsize(path), out["ratios"].ravel())


if __name__ == "__main__":
    main()
