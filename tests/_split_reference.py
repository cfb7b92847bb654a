"""Float64 references and bars for the split-precision DSAM backward (``DSAModule.grad_precision = "fp32"``).

The split kernels are held to the contraction of the EXACT fp32 operands (fp32 G, fp32 x * bit_t, fp32 weights), not to
the bf16 operands ``_grad_reference.dsam_reference`` rebuilds.  ``dsam_reference`` here is that same stage backward with
the rounding of the GEMM operands as a parameter: each product term names how G and the other operand (x for dW, the
weights for dx) are rounded, and the terms are summed.  Bias gradients and the identity residual are fp32 sums of fp32 G
in every mode and come from ``_grad_reference`` unchanged.

Error model: v = hi + lo + e with hi = bf16(v), lo = bf16(v - hi) (the fp32 subtraction is exact) and |e| <= 2^-16 |v|.
The three products hi.hi + lo.hi + hi.lo leave out lo.lo, e_a.b and hi_a.e_b, each at most 2^-16 |a||b|, so the
element-wise bar is (accumulation bar + TAU_SPLIT) * ref_abs with ref_abs the contraction over absolute values."""
from typing import Callable, Dict, Optional, Sequence, Tuple

import torch
from torch.nn.grad import conv2d_input, conv2d_weight

import _grad_reference as GR

TAU_SPLIT = 3 * 2.0 ** -16
# Relative L2 bar every split-precision check must also meet: the project's fp32 bar.  bf16 operands (~2^-8 each) can
# pass the element-wise bar once their errors average out over a long contraction, but not this one.
SPLIT_REL_L2 = 1e-4

Pair = Tuple[torch.Tensor, torch.Tensor]
Rounding = Callable[[torch.Tensor], torch.Tensor]


def hi_part(t: torch.Tensor) -> torch.Tensor:
    """bf16(v) widened to float64 (the hi part of the split)."""
    return GR.bf16(t)


def lo_part(t: torch.Tensor) -> torch.Tensor:
    """bf16(v - float(bf16(v))) widened to float64."""
    f = t.detach().float()
    return (f - f.to(torch.bfloat16).float()).to(torch.bfloat16).double()


def exact(t: torch.Tensor) -> torch.Tensor:
    """The fp32 operand itself, widened to float64."""
    return t.detach().float().double()


# (rounding of G, rounding of the other operand) per product term; the terms are summed
OPERANDS: Dict[str, Sequence[Tuple[Rounding, Rounding]]] = {
    "bf16": [(hi_part, hi_part)],                                           # what grad_precision "bf16" computes
    "fp32": [(exact, exact)],                                               # the exact fp32 operands
    "split": [(hi_part, hi_part), (lo_part, hi_part), (hi_part, lo_part)],  # float64 emulation of the split kernels
}


def _products(x, codes, g, params, R, g_round: Rounding, o_round: Rounding, dtype):
    """dW per weight name and dx (without the identity residual) of one product term, with their |.| contractions."""
    proj = "rgb_projection.weight" in params
    stride, pad = (2, 1) if proj else (1, 0)
    B = x.shape[0]
    bits = GR.region_bits(codes, R + 1).to(dtype)
    xr, gr = o_round(x).to(dtype), g_round(g).to(dtype)
    names = [f"conv_layers.{t}.weight" for t in range(R + 1)] + (["rgb_projection.weight"] if proj else [])
    c_out, c_in, k, _ = params["conv_layers.0.weight"].shape
    n_seg = len(names)
    # the mask commutes with both roundings (hi(0) = lo(0) = 0): segment t reads round(x) * bit_t
    xs = torch.cat([xr * bits[:, t:t + 1] for t in range(R + 1)] + ([xr] if proj else []), dim=1)
    dw = conv2d_weight(xs, (c_out, n_seg * c_in, k, k), gr, stride=stride, padding=pad)
    dwa = conv2d_weight(xs.abs(), (c_out, n_seg * c_in, k, k), gr.abs(), stride=stride, padding=pad)
    out = {name: (dw[:, s * c_in:(s + 1) * c_in], dwa[:, s * c_in:(s + 1) * c_in]) for s, name in enumerate(names)}
    ws = torch.cat([o_round(params[name]).to(dtype) for name in names], dim=1)
    shape = (B, n_seg * c_in) + tuple(x.shape[2:])
    dxs = conv2d_input(shape, ws, gr, stride=stride, padding=pad)
    dxsa = conv2d_input(shape, ws.abs(), gr.abs(), stride=stride, padding=pad)
    mask = torch.cat([bits[:, t:t + 1].expand(B, c_in, *x.shape[2:]) for t in range(R + 1)]
                     + ([torch.ones_like(xr)] if proj else []), dim=1)
    out["x"] = ((dxs * mask).reshape(B, n_seg, c_in, *x.shape[2:]).sum(1),
                (dxsa * mask).reshape(B, n_seg, c_in, *x.shape[2:]).sum(1))
    return out


def dsam_reference(x: torch.Tensor, codes: torch.Tensor, variant: Optional[torch.Tensor], g: torch.Tensor,
                   params: Dict[str, torch.Tensor], operands="fp32", num_regions: int = 3,
                   dtype=torch.float64) -> Dict[str, Pair]:
    """Backward of one DSAM stage (arguments as ``_grad_reference.dsam_reference``) with the GEMM operands rounded as
    ``operands`` says: "fp32" (the reference of the split kernels), "split" (a float64 emulation of them), "bf16", or a
    list of (G rounding, other rounding) product terms.  Returns {parameter name or "x": (ref, ref_abs)}."""
    terms = OPERANDS[operands] if isinstance(operands, str) else list(operands)
    x, g = x.detach().cpu(), g.detach().cpu()
    out: Dict[str, Pair] = {}
    for g_round, o_round in terms:
        for name, (r, ra) in _products(x, codes, g, params, num_regions, g_round, o_round, dtype).items():
            out[name] = (out[name][0] + r, out[name][1] + ra) if name in out else (r, ra)
    for t, pair in enumerate(GR.dsam_bias_reference(g, variant, num_regions + 1, dtype)):
        out[f"conv_layers.{t}.bias"] = pair
    if "rgb_projection.weight" not in params:             # identity residual: fp32 G, added once
        out["x"] = (out["x"][0] + g.to(dtype), out["x"][1] + g.to(dtype).abs())
    return out


def check_split(got: torch.Tensor, ref: torch.Tensor, ref_abs: torch.Tensor, tau: float) -> Dict:
    """The split-precision bar against the exact-operand reference: element-wise
    |got - ref| <= (tau + TAU_SPLIT) * ref_abs and relative L2 <= SPLIT_REL_L2."""
    res = GR.check(got, ref, ref_abs, tau + TAU_SPLIT)
    res["rel_l2_bar"] = SPLIT_REL_L2
    res["ok"] = res["ok"] and res["rel_l2"] <= SPLIT_REL_L2
    return res
