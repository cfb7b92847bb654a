"""State-dict layout (key -> shape, dtype) of the reference's depth-guidance modules -> tests/golden/state_dict_layout.json.

    python oracle/make_golden_layout.py

The tables are written from the weight factories (rgbd_b200.synthetic_weights).  The reference modules load those factories'
dicts with strict ``load_state_dict`` when oracle/make_golden*.py runs, and tests/test_host_logic.py compares the tables
with the live reference modules wherever the reference project is importable.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.make_golden import GOLD, load_pkg      # noqa: E402

# constructor call of the reference module -> the factory of its state dict
MODULES = {
    "DepthGradientInjectionResidual([96, 192, 384, 768], 3)": lambda W: W.dggm_weights([96, 192, 384, 768], 3, seed=0),
    "DSAModule(96, 192, 3)": lambda W: W.dsam_weights(96, 192, seed=0),
    "DSAModule(64, 64, 3)": lambda W: W.dsam_weights(64, 64, seed=0),
    "EnhancedDepthImageRatioPredictor(3)": lambda W: W.ratio_weights(seed=0),
}


def layout(state_dict) -> dict:
    return {k: {"shape": list(v.shape), "dtype": str(v.dtype).replace("torch.", "")} for k, v in state_dict.items()}


def main():
    _, weights = load_pkg()
    out = {name: layout(make(weights)) for name, make in MODULES.items()}
    path = os.path.join(GOLD, "state_dict_layout.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
