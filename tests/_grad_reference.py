"""Float64 references for the backward of one DSAM stage and of the DGGM 1x1 convs, and the element-wise checker the
backward tests share.

The references contract exactly the operands the CUDA kernels consume -- bf16 round-to-nearest of the output gradient G,
of x * bit_t(code) and of the weights; fp32 G for the bias gradient and the identity residual; the oracle's own fp32 gated
depth-gradient map for DGGM -- so they differ from a kernel only by its fp32 accumulation order.  Each result comes with
the same contraction taken over absolute values (``ref_abs``), which bounds that accumulation error element by element:
``|got - ref| <= tau * ref_abs``.  ``tests/test_grad_reference.py`` shows that this bar rejects the bugs it is meant to
catch (a dropped output column, a wrong tap, a wrong region bit, a wrong bias gate)."""
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F
from torch.nn.grad import conv2d_input, conv2d_weight

from oracle import hotpath as O

# Element-wise bars (relative to ref_abs), each more than 10x above the largest error measured on a B200 (1000 W) at the
# shapes of tests/test_gpu_backward.py (profiles/r03_parity_backward.jsonl): dW 1.3e-6 (Swin-B stage 0, K = 38 400 output
# pixels), dx 4.7e-7, DSAM db 4.3e-8, DGGM dW / db outside the gate band (see dggm_reference) 1.1e-7.
TAU_DW = 2e-5         # dsam_wgrad: tcgen05 products accumulated in tensor memory, split-K finished with fp32 atomics
TAU_DX = 1e-5         # the input-gradient GEMM (conv_gemm epilogue mode 3): fp32 accumulation + masked segment sum
TAU_DB = 1e-6         # DSAM bias gradients (fp32 sums of fp32 G)
TAU_DGGM = 1e-5       # DGGM dW / db (fp32 FMA chains and atomics)

Pair = Tuple[torch.Tensor, torch.Tensor]


def bf16(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 (round-to-nearest-even, like ``__float2bfloat16``) and widen to float64."""
    return t.detach().float().to(torch.bfloat16).double()


def region_bits(codes: torch.Tensor, n: int) -> torch.Tensor:
    """(B,H,W) uint8 codes -> (B,n,H,W) float64 0/1: bit t of every pixel."""
    c = codes.detach().cpu().to(torch.int32)
    return torch.stack([((c >> t) & 1) for t in range(n)], dim=1).double()


def dsam_bias_reference(g: torch.Tensor, variant: Optional[torch.Tensor], n_bias: int, dtype=torch.float64):
    """[(db_t, db_t over |G|)] for t < n_bias: db_t = sum over the images that add bias t (t < variant[b]; all images
    when variant is None) and over all output pixels of fp32 G, without rounding."""
    g = g.detach().cpu()
    v = torch.full((g.shape[0],), n_bias) if variant is None else variant.detach().cpu().long()
    gs = g.to(dtype).sum(dim=(2, 3))                                       # (B, C_out)
    gsa = g.to(dtype).abs().sum(dim=(2, 3))
    out = []
    for t in range(n_bias):
        use = (t < v).to(dtype)[:, None]
        out.append(((gs * use).sum(0), (gsa * use).sum(0)))
    return out


def dsam_reference(x: torch.Tensor, codes: torch.Tensor, variant: Optional[torch.Tensor], g: torch.Tensor,
                   params: Dict[str, torch.Tensor], num_regions: int = 3, dtype=torch.float64) -> Dict[str, Pair]:
    """Backward of one DSAM stage.  x (B,C_in,H,W) fp32, codes (B,H,W) uint8 at the stage input's resolution (bit t =
    region mask t, ``Decomposition.pooled[k]``), variant (B,) = number of conv biases image b adds (None: all), g
    (B,C_out,Ho,Wo) fp32, params = the module's fp32 weights by parameter name.  Returns {parameter name or "x":
    (ref, ref_abs)} in ``dtype`` (float32 models a kernel that differs only in its summation order).  The projection
    variant (``rgb_projection.weight`` present) is a 3x3 stride-2 pad-1 conv, the identity variant a 1x1 conv plus the
    residual F."""
    R = num_regions
    proj = "rgb_projection.weight" in params
    stride, pad = (2, 1) if proj else (1, 0)
    x = x.detach().cpu()
    g = g.detach().cpu()
    B = x.shape[0]
    bits = region_bits(codes, R + 1).to(dtype)                             # (B, R+1, H, W)
    xb, gb = bf16(x).to(dtype), bf16(g).to(dtype)
    ga = gb.abs()
    out: Dict[str, Pair] = {}

    # dW: every segment in one contraction over (B, Ho, Wo); segment t reads bf16(x * bit_t) = bit_t * bf16(x)
    segs_x = [xb * bits[:, t:t + 1] for t in range(R + 1)] + ([xb] if proj else [])
    n_seg = len(segs_x)
    c_out, c_in, k, _ = params["conv_layers.0.weight"].shape
    xs = torch.cat(segs_x, dim=1)
    dw = conv2d_weight(xs, (c_out, n_seg * c_in, k, k), gb, stride=stride, padding=pad)
    dwa = conv2d_weight(xs.abs(), (c_out, n_seg * c_in, k, k), ga, stride=stride, padding=pad)
    names = [f"conv_layers.{t}.weight" for t in range(R + 1)] + (["rgb_projection.weight"] if proj else [])
    for s, name in enumerate(names):
        out[name] = (dw[:, s * c_in:(s + 1) * c_in], dwa[:, s * c_in:(s + 1) * c_in])

    for t, pair in enumerate(dsam_bias_reference(g, variant, R + 1, dtype)):
        out[f"conv_layers.{t}.bias"] = pair

    # dx = sum_t bit_t * ConvT_t(bf16 G) + ProjT(bf16 G)  [identity variant: + fp32 G]
    ws = torch.cat([bf16(params[name]).to(dtype) for name in names], dim=1)        # (C_out, n_seg*C_in, k, k)
    shape = (B, n_seg * c_in) + tuple(x.shape[2:])
    dxs = conv2d_input(shape, ws, gb, stride=stride, padding=pad)
    dxsa = conv2d_input(shape, ws.abs(), ga, stride=stride, padding=pad)
    mask = torch.cat([bits[:, t:t + 1].expand(B, c_in, *x.shape[2:]) for t in range(R + 1)]
                     + ([torch.ones_like(xb)] if proj else []), dim=1)
    dx = (dxs * mask).reshape(B, n_seg, c_in, *x.shape[2:]).sum(1)
    dxa = (dxsa * mask).reshape(B, n_seg, c_in, *x.shape[2:]).sum(1)
    if not proj:
        dx = dx + g.to(dtype)
        dxa = dxa + g.to(dtype).abs()
    out["x"] = (dx, dxa)
    return out


# fraction of |b| + sum_d |w_d * gated_d| inside which the sign of the DGGM pre-activation is not fixed by fp32 arithmetic
# (the kernel's gated map may differ from the oracle's by an ulp: FMA contraction of the bilinear weights)
GATE_BAND = 1e-6


def dggm_reference(w: Dict[str, torch.Tensor], grad: torch.Tensor, mask: torch.Tensor,
                   douts: Sequence[torch.Tensor]) -> Dict[str, Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]:
    """Parameter gradients of ``DepthGradientInjectionResidual``: dW_i[c,d] = sum relu'(e) * dout * gated_d and
    db_i[c] = sum relu'(e) * dout in float64, where ``gated`` is the oracle's fp32 bilinear(grad) * nearest(mask)
    (exactly as ``oracle.hotpath.dggm_forward`` builds it) and the gate is e > 0 for the pre-activation e = W gated + b.
    Returns {name: (ref, ref_abs, slack)}: ``slack`` is the absolute contraction over the pixels whose |e| lies within
    GATE_BAND of its own magnitude, where fp32 rounding alone may flip the gate.  Such flips happen: at 480x640, B = 8
    one pixel of one channel of the 60x80 scale flips and moves dW of that channel by 1.1e-4 of ref_abs -- the whole of
    that pixel's term -- while every element stays within 1.1e-7 of ref_abs outside the band."""
    out = {}
    grad_np, mask_np = grad.detach().cpu().numpy(), mask.detach().cpu().numpy()
    for i, d in enumerate(douts):
        hw = tuple(d.shape[2:])
        gm = torch.from_numpy(O.bilinear_downsample(grad_np, hw))
        mm = torch.from_numpy(np.ascontiguousarray(O.nearest_downsample(mask_np, hw)))
        gated = (gm * mm).double()                                          # fp32 product, as the oracle forms it
        wi = w[f"depth_enhancement_layers.{i}.0.weight"].detach().cpu().double()
        bi = w[f"depth_enhancement_layers.{i}.0.bias"].detach().cpu().double()
        e = F.conv2d(gated, wi, bi)
        mag = F.conv2d(gated.abs(), wi.abs(), bi.abs())
        amb = (e.abs() <= GATE_BAND * mag).double()
        on = (e > 0).double()
        do = d.detach().cpu().double()
        gd, gda = do * on, do.abs() * on
        ga = do.abs() * amb
        dw = torch.einsum("bchw,bdhw->cd", gd, gated)[:, :, None, None]
        dwa = torch.einsum("bchw,bdhw->cd", gda, gated.abs())[:, :, None, None]
        dws = torch.einsum("bchw,bdhw->cd", ga, gated.abs())[:, :, None, None]
        out[f"depth_enhancement_layers.{i}.0.weight"] = (dw, dwa, dws)
        out[f"depth_enhancement_layers.{i}.0.bias"] = (gd.sum((0, 2, 3)), gda.sum((0, 2, 3)), ga.sum((0, 2, 3)))
    return out


def check(got: torch.Tensor, ref: torch.Tensor, ref_abs: torch.Tensor, tau: float,
          slack: Optional[torch.Tensor] = None) -> Dict:
    """Element-wise bar |got - ref| <= tau * ref_abs + slack + 1e-30 (an element whose every term is zero must come out
    exactly zero).  Returns {"ok", "n_bad", "max_norm_err" (largest |got - ref| / ref_abs), "rel_l2", "tau"}."""
    got = got.detach().double().cpu()
    if tuple(got.shape) != tuple(ref.shape):
        return {"ok": False, "n_bad": -1, "max_norm_err": float("inf"), "rel_l2": float("inf"), "tau": tau,
                "shape": [list(got.shape), list(ref.shape)]}
    err = (got - ref).abs()
    bound = tau * ref_abs + 1e-30
    if slack is not None:
        bound = bound + slack
    bad = ~(err <= bound)                                                  # NaN counts as bad
    def max_norm(e):
        n = torch.where(ref_abs > 0, e / ref_abs.clamp_min(1e-300), torch.where(e > 0, torch.inf, 0.0))
        return float(n.max()) if n.numel() else 0.0
    res = {"ok": not bool(bad.any()), "n_bad": int(bad.sum()), "max_norm_err": max_norm(err),
           "rel_l2": float(err.norm() / ref.norm().clamp_min(1e-300)), "tau": tau}
    if slack is not None:
        res["max_norm_err_outside_slack"] = max_norm((err - slack).clamp_min(0.0))
    return res


def tau_for(name: str) -> float:
    """Bar of a DSAM parameter name, "x" (the stage input) or a DGGM parameter name."""
    if name == "x":
        return TAU_DX
    if name.startswith("depth_enhancement_layers."):
        return TAU_DGGM
    return TAU_DB if name.endswith(".bias") else TAU_DW
