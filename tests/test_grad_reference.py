"""The float64 backward references of tests/_grad_reference.py, checked on the CPU: they equal torch autograd through the
oracle (``oracle.hotpath.dsam_forward`` / ``dggm_forward``) in float64 on the same pre-rounded operands, and the
element-wise bar the GPU backward tests apply rejects "kernel outputs" that carry the bugs a backward kernel is prone to,
at the benchmarked reduction length (120x160 stage input, B = 8: K = B*Ho*Wo = 38 400)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rgbd_b200  # noqa: F401
from rgbd_b200 import synthetic
from oracle import hotpath as O
from oracle import weights as OW
import _grad_reference as GR


def _gray(idx, kind, dhw):
    _, d = synthetic.synth_rgbd_u8(idx, dhw[0], dhw[1], kind)
    return O.to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))


def _oracle_codes(gray, ratio, hw):
    """Pooled region codes and bias variant exactly as oracle.hotpath.dsam_forward derives its masks."""
    masks = O.depth_decompose(gray, ratio)["masks"]
    codes = np.zeros(hw, dtype=np.uint8)
    for t, m in enumerate(masks):
        codes |= O.adaptive_max_pool_mask(m, hw).astype(np.uint8) << t
    return codes, len(masks)


def _autograd_case(ci, co, hw, dhw, frames, seed):
    w = OW.dsam_weights(ci, co, seed=seed)
    rs = np.random.RandomState(seed)
    B = len(frames)
    grays = [_gray(idx, kind, dhw) for idx, kind in frames]
    ratios = [0.1, 0.3, 0.2, 0.4][:B]
    cv = [_oracle_codes(g, r, hw) for g, r in zip(grays, ratios)]
    codes = torch.from_numpy(np.stack([c for c, _ in cv]))
    variant = torch.tensor([v for _, v in cv], dtype=torch.int32)
    x = torch.from_numpy(rs.randn(B, ci, *hw).astype(np.float32))
    return w, grays, ratios, codes, variant, x


@pytest.mark.parametrize("ci,co,hw,dhw,frames", [
    (40, 72, (13, 17), (52, 68), [(20, "nyu"), (21, "constant"), (22, "uniform")]),     # odd H/W, C_in % 32 != 0
    (32, 64, (12, 16), (96, 128), [(20, "nyu"), (23, "two_valued")]),
    (24, 24, (9, 11), (36, 44), [(22, "uniform"), (21, "constant"), (20, "nyu")]),        # identity 1x1 variant
], ids=["proj-odd-40to72", "proj-32to64", "identity-24"])
def test_dsam_reference_equals_float64_oracle_autograd(ci, co, hw, dhw, frames):
    w, grays, ratios, codes, variant, x = _autograd_case(ci, co, hw, dhw, frames, seed=400 + ci + co)
    if any(kind == "constant" for _, kind in frames):          # one depth mode: the image adds 2 of the 4 biases
        assert int(variant.min()) < 4
    B = x.shape[0]
    proj = ci != co
    Ho, Wo = ((hw[0] + 1) // 2, (hw[1] + 1) // 2) if proj else hw
    g = torch.from_numpy(np.random.RandomState(7).randn(B, co, Ho, Wo).astype(np.float32))
    ref = GR.dsam_reference(x, codes, variant, g, w)

    # autograd through the oracle in float64 on the operands the kernels see: bf16 weights / x / G, fp32 G for the biases
    wr = {k: (GR.bf16(v) if k.endswith("weight") else v.double()).requires_grad_(True) for k, v in w.items()}
    xr = GR.bf16(x).requires_grad_(True)
    out = torch.cat([O.dsam_forward(wr, xr[b:b + 1], grays[b], ratios[b]) for b in range(B)])
    gb, g64 = GR.bf16(g), g.double()
    wnames = [k for k in w if k.endswith("weight")]
    bnames = [k for k in w if k.endswith("bias")]
    gw = torch.autograd.grad((out * gb).sum(), [wr[k] for k in wnames] + [xr], retain_graph=True, allow_unused=True)
    gbias = torch.autograd.grad((out * g64).sum(), [wr[k] for k in bnames], allow_unused=True)
    auto = dict(zip(wnames + ["x"], gw))
    auto.update(zip(bnames, gbias))
    if not proj:                  # the identity residual: autograd passed bf16(G) through it, the kernels pass fp32 G
        auto["x"] = auto["x"] - gb + g64
    assert set(ref) == set(auto)
    for name, (r, ra) in ref.items():
        a = auto[name]
        if a is None:             # segment no image uses: the oracle leaves no gradient, the reference is exactly zero
            assert float(ra.abs().max()) == 0.0 and float(r.abs().max()) == 0.0, name
            continue
        res = GR.check(a, r, ra, 1e-12)
        assert res["ok"], (name, res)


@pytest.mark.parametrize("chans,hw,sizes,B", [
    ([8, 16, 24, 32], (64, 96), [(16, 24), (8, 12), (4, 6), (2, 3)], 2),
    ([4, 8, 12, 16], (50, 70), [(13, 18), (7, 9), (4, 5), (2, 3)], 3),
])
def test_dggm_reference_equals_float64_oracle_autograd(monkeypatch, chans, hw, sizes, B):
    rs = np.random.RandomState(31)
    w = OW.dggm_weights(chans, 3, seed=302)
    feats = [torch.from_numpy(rs.randn(B, c, h, ww)) for c, (h, ww) in zip(chans, sizes)]       # float64
    grad = torch.from_numpy(rs.rand(B, 3, *hw).astype(np.float32))
    mask = torch.from_numpy((rs.rand(B, 1, *hw) < 0.6).astype(np.float32))
    douts = [torch.from_numpy(rs.randn(*f.shape).astype(np.float32)) for f in feats]
    ref = GR.dggm_reference(w, grad, mask, douts)
    # the oracle forms the gated map in float32 (as the kernel does); widen it to float64 at the 1x1 conv
    conv2d = F.conv2d
    monkeypatch.setattr(F, "conv2d", lambda inp, wt, b=None, **kw: conv2d(inp.to(wt.dtype), wt, b, **kw))
    wr = {k: v.double().requires_grad_(True) for k, v in w.items()}
    out = O.dggm_forward(wr, feats, grad, mask)
    sum((o * d.double()).sum() for o, d in zip(out, douts)).backward()
    for name, (r, ra, slack) in ref.items():
        res = GR.check(wr[name].grad, r, ra, 1e-12)
        assert res["ok"], (name, res)


# ---------------------------------------------------------------------------------------------------
# the bar rejects the bugs it is meant to catch
# ---------------------------------------------------------------------------------------------------
def _mutation_case():
    """120x160 stage input, B = 8 (Swin-T stage 0 at 480x640), narrow channels; region codes with every bit pattern
    and per-image bias variants 1..4."""
    rs = np.random.RandomState(11)
    B, ci, co, (H, W) = 8, 8, 16, (120, 160)
    w = OW.dsam_weights(ci, co, seed=500)
    variant = torch.tensor([4, 2, 3, 4, 1, 4, 2, 3], dtype=torch.int32)
    codes = np.zeros((B, H, W), dtype=np.uint8)
    for b in range(B):
        for t in range(int(variant[b])):
            codes[b] |= (rs.rand(H, W) < 0.45).astype(np.uint8) << t
    x = torch.from_numpy(rs.randn(B, ci, H, W).astype(np.float32))
    g = torch.from_numpy(rs.randn(B, co, H // 2, W // 2).astype(np.float32))
    return w, torch.from_numpy(codes), variant, x, g


def _shift_right(t, n):
    """t[..., j] -> t[..., j - n] (zero fill): the packed plane the x-1 taps read, one parity-plane pixel off."""
    return F.pad(t, (n, 0))[..., :t.shape[-1]]


def _mutations(w, codes, variant, x, g, base):
    """name -> (mutated {tensor name: kernel output}, tensor names that must fail the bar)."""
    ref = lambda **kw: {k: v[0] for k, v in GR.dsam_reference(  # noqa: E731
        kw.get("x", x), kw.get("codes", codes), variant, kw.get("g", g), kw.get("w", w)).items()}
    muts = {}
    weights = [f"conv_layers.{t}.weight" for t in range(4)] + ["rgb_projection.weight"]

    g2 = g.clone()
    g2[..., -1] = 0
    muts["g_last_output_column_zeroed"] = (ref(g=g2), weights + ["conv_layers.0.bias", "x"])

    g2 = g.clone()
    g2[5] = 0
    muts["one_image_g_zeroed"] = (ref(g=g2), weights + ["conv_layers.0.bias", "x"])

    got = {k: v.clone() for k, v in base.items()}
    for k in weights:
        got[k][..., 0, [0, 2]] = got[k][..., 0, [2, 0]]
    ws = {k: v.clone() for k, v in w.items()}
    for k in weights:
        ws[k][..., 0, [0, 2]] = ws[k][..., 0, [2, 0]]
    got["x"] = ref(w=ws)["x"]
    muts["taps_00_02_swapped"] = (got, weights + ["x"])

    got = {k: v.clone() for k, v in base.items()}
    off = ref(x=_shift_right(x, 2), codes=_shift_right(codes, 2))
    for k in weights:
        got[k][..., 0] = off[k][..., 0]
    muts["x_minus_1_taps_one_pixel_off"] = (got, weights)

    c2 = (codes & 0xFD) | ((codes >> 1) & 2)                               # segment 1 reads bit 2
    muts["segment_1_reads_region_bit_2"] = (ref(codes=c2), ["conv_layers.1.weight", "x"])

    got = {k: v.clone() for k, v in base.items()}
    use = (variant.long() > 2).double()[:, None]                           # bias 1 gated by variant > t+1
    got["conv_layers.1.bias"] = (g.double().sum((2, 3)) * use).sum(0)
    muts["bias_1_gated_by_variant_gt_2"] = (got, ["conv_layers.1.bias"])
    return muts


@pytest.fixture(scope="module")
def mutation_case():
    w, codes, variant, x, g = _mutation_case()
    full = GR.dsam_reference(x, codes, variant, g, w)
    muts = _mutations(w, codes, variant, x, g, {k: v[0] for k, v in full.items()})
    return w, codes, variant, x, g, full, muts


def test_the_bar_accepts_a_reordered_fp32_computation(mutation_case):
    """Positive control: the same contractions accumulated in float32 (a different summation order, as a kernel has)
    pass at the bars the GPU tests use."""
    w, codes, variant, x, g, full, _ = mutation_case
    f32 = GR.dsam_reference(x, codes, variant, g, w, dtype=torch.float32)
    for name, (r, ra) in full.items():
        res = GR.check(f32[name][0], r, ra, GR.tau_for(name))
        assert res["ok"], (name, res)
        assert res["max_norm_err"] < GR.tau_for(name) / 10, (name, res)


@pytest.mark.parametrize("mutation", ["g_last_output_column_zeroed", "one_image_g_zeroed", "taps_00_02_swapped",
                                      "x_minus_1_taps_one_pixel_off", "segment_1_reads_region_bit_2",
                                      "bias_1_gated_by_variant_gt_2"])
def test_the_bar_rejects_a_mutated_backward(mutation_case, mutation):
    full, muts = mutation_case[5], mutation_case[6]
    got, must_fail = muts[mutation]
    for name in must_fail:
        r, ra = full[name]
        res = GR.check(got[name], r, ra, GR.tau_for(name))
        assert not res["ok"], (mutation, name, res)
        print(mutation, name, res)
