"""The references of the split-precision DSAM backward (``DSAModule.grad_precision = "fp32"``), checked on the CPU.

The split-precision kernels are held to the contraction of the exact fp32 operands (fp32 G, fp32 x * bit_t, fp32
weights; ``_split_reference.dsam_reference(operands="fp32")``) at an analytic element-wise bar (TAU_SPLIT = 3 * 2^-16 on
top of the accumulation bar) and at relative L2 1e-4.  Here: with bf16 operands it reproduces
``_grad_reference.dsam_reference``; with the exact operands it equals float64 autograd through the oracle; a
float64 emulation of the three-product split meets both bars at the benchmarked reduction length; the bf16-operand
computation and the split with either cross product dropped fail them; and the split weight tables of
``DSAModule._refresh_bwd``, contracted by a GEMM emulation, reproduce the exact-operand input gradient."""
import numpy as np
import pytest
import torch

import rgbd_b200  # noqa: F401
from rgbd_b200 import modules, synthetic
from oracle import hotpath as O
from oracle import weights as OW
import _grad_reference as GR
import _split_reference as SR


def _autograd_case(ci, co, hw, dhw, frames, seed):
    """Weights, grays, ratios, pooled region codes and bias variants exactly as oracle.hotpath.dsam_forward derives its
    masks, and a random stage input."""
    w = OW.dsam_weights(ci, co, seed=seed)
    rs = np.random.RandomState(seed)
    grays, codes, variant = [], [], []
    ratios = [0.1, 0.3, 0.2, 0.4][:len(frames)]
    for (idx, kind), r in zip(frames, ratios):
        _, d = synthetic.synth_rgbd_u8(idx, dhw[0], dhw[1], kind)
        gray = O.to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
        masks = O.depth_decompose(gray, r)["masks"]
        c = np.zeros(hw, dtype=np.uint8)
        for t, m in enumerate(masks):
            c |= O.adaptive_max_pool_mask(m, hw).astype(np.uint8) << t
        grays.append(gray)
        codes.append(c)
        variant.append(len(masks))
    x = torch.from_numpy(rs.randn(len(frames), ci, *hw).astype(np.float32))
    return w, grays, ratios, torch.from_numpy(np.stack(codes)), torch.tensor(variant, dtype=torch.int32), x


_AUTOGRAD_CASES = [
    (40, 72, (13, 17), (52, 68), [(20, "nyu"), (21, "constant"), (22, "uniform")]),     # projection, odd H/W
    (24, 24, (9, 11), (36, 44), [(22, "uniform"), (21, "constant"), (20, "nyu")]),        # identity 1x1 variant
]


@pytest.mark.parametrize("ci,co,hw,dhw,frames", _AUTOGRAD_CASES, ids=["proj-odd-40to72", "identity-24"])
def test_bf16_operands_reproduce_the_bf16_backward_reference(ci, co, hw, dhw, frames):
    """``_split_reference.dsam_reference(operands="bf16")`` is ``_grad_reference.dsam_reference``: same tensors, same
    values (<= 1e-12 of ref_abs), so the two modules rebuild the stage backward the same way."""
    w, _, _, codes, variant, x = _autograd_case(ci, co, hw, dhw, frames, seed=460 + ci + co)
    Ho, Wo = ((hw[0] + 1) // 2, (hw[1] + 1) // 2) if ci != co else hw
    g = torch.from_numpy(np.random.RandomState(9).randn(x.shape[0], co, Ho, Wo).astype(np.float32))
    ours = SR.dsam_reference(x, codes, variant, g, w, operands="bf16")
    base = GR.dsam_reference(x, codes, variant, g, w)
    assert set(ours) == set(base)
    for name, (r, ra) in base.items():
        assert GR.check(ours[name][0], r, ra, 1e-12)["ok"], name
        assert GR.check(ours[name][1], ra, ra, 1e-12)["ok"], name


@pytest.mark.parametrize("ci,co,hw,dhw,frames", _AUTOGRAD_CASES, ids=["proj-odd-40to72", "identity-24"])
def test_fp32_operand_reference_equals_float64_oracle_autograd(ci, co, hw, dhw, frames):
    w, grays, ratios, codes, variant, x = _autograd_case(ci, co, hw, dhw, frames, seed=450 + ci + co)
    B = x.shape[0]
    proj = ci != co
    Ho, Wo = ((hw[0] + 1) // 2, (hw[1] + 1) // 2) if proj else hw
    g = torch.from_numpy(np.random.RandomState(8).randn(B, co, Ho, Wo).astype(np.float32))
    ref = SR.dsam_reference(x, codes, variant, g, w, operands="fp32")
    wr = {k: v.double().requires_grad_(True) for k, v in w.items()}
    xr = x.double().requires_grad_(True)
    out = torch.cat([O.dsam_forward(wr, xr[b:b + 1], grays[b], ratios[b]) for b in range(B)])
    (out * g.double()).sum().backward()
    for name, (r, ra) in ref.items():
        a = xr.grad if name == "x" else wr[name].grad
        if a is None:             # segment no image uses: the oracle leaves no gradient, the reference is exactly zero
            assert float(ra.abs().max()) == 0.0 and float(r.abs().max()) == 0.0, name
            continue
        res = GR.check(a, r, ra, 1e-12)
        assert res["ok"], (name, res)


# ---------------------------------------------------------------------------------------------------
# the split bars accept the split and reject what is not the split, at Swin-T stage 0 of the train record
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def swin_t_s0():
    """120x160 stage input, B = 8, 96 -> 192 channels (Swin-T stage 0 at 480x640): K = 38 400 output pixels for dW.
    Region codes with every bit pattern, per-image bias variants 1..4.  Returns the exact-operand reference and the
    three products of the split as separate contractions (hi.hi alone is the bf16 mode)."""
    rs = np.random.RandomState(12)
    B, ci, co, (H, W) = 8, 96, 192, (120, 160)
    w = OW.dsam_weights(ci, co, seed=501)
    variant = torch.tensor([4, 2, 3, 4, 1, 4, 2, 3], dtype=torch.int32)
    codes = np.zeros((B, H, W), dtype=np.uint8)
    for b in range(B):
        for t in range(int(variant[b])):
            codes[b] |= (rs.rand(H, W) < 0.45).astype(np.uint8) << t
    codes = torch.from_numpy(codes)
    x = torch.from_numpy(rs.randn(B, ci, H, W).astype(np.float32))
    g = torch.from_numpy(rs.randn(B, co, H // 2, W // 2).astype(np.float32))
    ref = SR.dsam_reference(x, codes, variant, g, w, operands="fp32")
    terms = {name: {k: v[0] for k, v in SR.dsam_reference(x, codes, variant, g, w, operands=[t]).items()}
             for name, t in (("hi_hi", (SR.hi_part, SR.hi_part)), ("lo_hi", (SR.lo_part, SR.hi_part)),
                             ("hi_lo", (SR.hi_part, SR.lo_part)))}
    return ref, terms


_GEMM_TENSORS = [f"conv_layers.{t}.weight" for t in range(4)] + ["rgb_projection.weight", "x"]


def _tau(name):
    return GR.TAU_DX if name == "x" else GR.TAU_DW


def test_split_emulation_meets_both_bars(swin_t_s0):
    ref, terms = swin_t_s0
    for name in _GEMM_TENSORS:
        got = terms["hi_hi"][name] + terms["lo_hi"][name] + terms["hi_lo"][name]
        res = SR.check_split(got, *ref[name], _tau(name))
        assert res["ok"], (name, res)
        print("split", name, res)


@pytest.mark.parametrize("variant,products", [
    ("bf16_operands", ("hi_hi",)),               # what grad_precision "bf16" computes
    ("x_lo_w_hi_dropped", ("hi_hi", "hi_lo")),   # G_lo . X_hi / G_lo . W_hi missing
    ("x_hi_w_lo_dropped", ("hi_hi", "lo_hi")),   # G_hi . X_lo / G_hi . W_lo missing
])
def test_split_bars_reject_what_is_not_the_split(swin_t_s0, variant, products):
    ref, terms = swin_t_s0
    for name in _GEMM_TENSORS:
        got = sum(terms[p][name] for p in products)
        res = SR.check_split(got, *ref[name], _tau(name))
        assert not res["ok"], (variant, name, res)
        assert res["rel_l2"] > SR.SPLIT_REL_L2, (variant, name, res)
        print(variant, name, res)


# ---------------------------------------------------------------------------------------------------
# the split tables of _refresh_bwd
# ---------------------------------------------------------------------------------------------------
def _emu_conv_gemm(a, plane_per_img, w, slices, kb, n_img, out_hw):
    """Float64 model of rgbd_conv_gemm's K loop.  a: (planes, Y, X, C); w: (N, n_slices*kb); slice (c0, dx, dy, plane)
    reads a[img * plane_per_img + plane, y + dy, x + dx, c0:c0 + kb], zero outside the tensor (TMA fill)."""
    planes, Y, X, Cc = a.shape
    Ho, Wo = out_hw
    ap = np.zeros((planes, Y + 4, X + 4, Cc), np.float64)
    ap[:, 2:2 + Y, 2:2 + X] = a
    out = np.zeros((n_img, Ho, Wo, w.shape[0]), np.float64)
    for j, (c0, dx, dy, dp) in enumerate(slices):
        wj = w[:, j * kb:(j + 1) * kb].T
        for img in range(n_img):
            src = ap[img * plane_per_img + dp, 2 + dy:2 + dy + Ho, 2 + dx:2 + dx + Wo, c0:c0 + kb]
            out[img, :src.shape[0], :src.shape[1]] += src @ wj
    return out


@pytest.mark.parametrize("ci,co,hw,B", [(40, 72, (15, 21), 2), (96, 192, (12, 16), 2), (24, 24, (9, 11), 2)],
                         ids=["proj-odd-40to72", "proj-96to192", "identity-24"])
def test_split_backward_tables_reproduce_the_fp32_input_gradient(ci, co, hw, B):
    rs = np.random.RandomState(ci + co)
    w = OW.dsam_weights(ci, co, seed=7)
    m = modules.DSAModule(ci, co, 3)
    m.load_state_dict(w)
    m.grad_precision = "fp32"
    pk = m._refresh_bwd()
    assert pk["split"]
    proj = ci != co
    H, W = hw
    Ho, Wo = ((H + 1) // 2, (W + 1) // 2) if proj else hw
    n_seg, np64 = pk["n_seg"], pk["np64"]
    codes = torch.from_numpy((rs.rand(B, H, W) * 16).astype(np.uint8))
    x = torch.from_numpy(rs.randn(B, ci, H, W).astype(np.float32))
    g = torch.from_numpy(rs.randn(B, co, Ho, Wo).astype(np.float32))
    # G channels-last, planes (hi, lo) per image: rgbd_dsam_pack(n_seg=1, hi_lo=1)
    a = np.zeros((B, 2, Ho, Wo, np64))
    a[:, 0, ..., :co] = SR.hi_part(g).permute(0, 2, 3, 1).numpy()
    a[:, 1, ..., :co] = SR.lo_part(g).permute(0, 2, 3, 1).numpy()
    a = a.reshape(B * 2, Ho, Wo, np64)
    bits = GR.region_bits(codes, 4).numpy()
    dx = np.zeros((B, ci, H, W))
    for cl in pk["classes"]:
        py, px = cl["py"], cl["px"]
        H2, W2 = ((H - py + 1) // 2, (W - px + 1) // 2) if proj else (H, W)
        wt = cl["w"].float().numpy()
        assert wt.shape[1] == cl["slices"].shape[0] * 64
        out = _emu_conv_gemm(a, 2, wt, cl["slices"].numpy().tolist(), 64, B, (H2, W2))
        out = out.reshape(B, H2, W2, -1, n_seg, 32)                 # columns: (channel block, segment, 32 channels)
        out = out.transpose(0, 3, 5, 4, 1, 2).reshape(B, -1, n_seg, H2, W2)[:, :ci]
        sy, sx = (slice(py, None, 2), slice(px, None, 2)) if proj else (slice(None), slice(None))
        mask = np.concatenate([bits[:, :, sy, sx], np.ones((B, n_seg - 4, H2, W2))], axis=1)   # projection: unmasked
        dx[:, :, sy, sx] = (out * mask[:, None]).sum(2)
    if not proj:
        dx = dx + g.double().numpy()                                 # identity residual: fp32 G
    r, ra = SR.dsam_reference(x, codes, None, g, w, operands="fp32")["x"]
    res = GR.check(torch.from_numpy(dx), r, ra, SR.TAU_SPLIT)
    assert res["ok"], res
    assert res["rel_l2"] <= SR.SPLIT_REL_L2, res


def test_grad_precision_accepts_only_bf16_and_fp32():
    m = modules.DSAModule(8, 16, 3)
    assert m.grad_precision == "bf16"
    m.grad_precision = "fp16"
    with pytest.raises(ValueError):
        m._refresh_bwd()
    with pytest.raises(ValueError):
        modules.DepthGuidance((8, 16, 24, 32), grad_precision="fp16")
    g = modules.DepthGuidance((8, 16, 24, 32), grad_precision="fp32")
    assert [d.grad_precision for d in (g.dsam0, g.dsam1, g.dsam2)] == ["fp32"] * 3
    assert [d.precision for d in (g.dsam0, g.dsam1, g.dsam2)] == ["bf16"] * 3
